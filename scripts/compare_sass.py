"""Compare the machine code of every kernel in two builds of libldeq.so.

    python scripts/compare_sass.py OLD/libldeq.so NEW/libldeq.so

A refactor of the host code that picks and launches kernels must leave every kernel's instructions as they were.  This
dumps both libraries with `cuobjdump -sass`, splits the dumps by `Function :`, strips the addresses and encodings, and
compares each kernel with its counterpart: the kernel of the same (demangled) name, the n-th copy matched with the n-th
when a name occurs more than once (a kernel defined in two translation units).  The Tsit5 kernels that once had their
own names are matched under their current ones: tsit5_fwd_kernel<RHS, S, TAPE> is erk_fwd_kernel<Tsit5M, RHS, S, TAPE>,
tsit5_bwd_kernel likewise, and tsit5_fwdsens_kernel<S, NP, FRICTION, SEED_P> is erk_fwdsens_kernel<Tsit5Dual, ...>.
Exits 1 on any difference.
"""
import collections
import os
import re
import subprocess
import sys

CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
RENAMED = [("ldeq::tsit5_fwd_kernel<", "ldeq::erk_fwd_kernel<ldeq::Tsit5M, "),
           ("ldeq::tsit5_bwd_kernel<", "ldeq::erk_bwd_kernel<ldeq::Tsit5M, "),
           ("ldeq::tsit5_fwdsens_kernel<", "ldeq::erk_fwdsens_kernel<ldeq::Tsit5Dual, ")]


def kernels(lib):
    """{(demangled name, copy index): instruction text} in dump order."""
    dump = subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-sass", lib], check=True, capture_output=True, text=True).stdout
    parts = re.split(r"^\s*Function : (\S+)\s*$", dump, flags=re.M)
    names = parts[1::2]
    plain = subprocess.run(["c++filt"], input="\n".join(names), check=True, capture_output=True, text=True).stdout.split("\n")
    out, seen = {}, collections.Counter()
    for name, body in zip(plain, parts[2::2]):
        for old, new in RENAMED:
            name = name.replace(old, new)
        lines = []
        for ln in body.split("\n"):
            ln = ln.strip()
            m = re.match(r"/\*[0-9a-f]{4,}\*/(.*?)(/\*\s*0x[0-9a-f]+\s*\*/)?$", ln)   # /*addr*/ instruction /* encoding */
            if m:
                lines.append(" ".join(m.group(1).split()))
            elif ln.startswith(".headerflags"):
                lines.append(ln)
        out[(name, seen[name])] = "\n".join(lines)
        seen[name] += 1
    return out


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    print(f"{len(old)} kernels in {sys.argv[1]}, {len(new)} in {sys.argv[2]}")
    bad = 0
    for key in sorted(set(old) | set(new)):
        if key not in old or key not in new:
            print(("only in new: " if key in new else "only in old: ") + f"{key[0]} #{key[1]}")
            bad += 1
        elif old[key] != new[key]:
            print(f"differs: {key[0]} #{key[1]}")
            bad += 1
    same = len(set(old) & set(new)) - sum(1 for k in set(old) & set(new) if old[k] != new[k])
    print(f"{same} identical, {bad} different or unmatched")
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
