"""CPU oracle for the LatentDiffEq.jl hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this package.  The product (``latentdiffeq.jl_b200`` and
``libldeq.so``) never imports, links or executes anything in here.

PARITY UNPINNED: the reference (gabrevaya/LatentDiffEq.jl) ships no tests, golden vectors or
stored outputs (``test/runtests.jl:4-6`` is an empty test set) and Julia is not available in this
image, so the oracle restates the published algorithms of the pinned third-party Julia packages
(SURVEY.md Appendix A) and is pinned by independent checks in ``tests/`` instead.

Modules
-------
goku   ctypes front-end of ``libldeq_oracle.so`` (C++/OpenMP): per-trajectory Tsit5 ensemble solve
       and ForwardDiffSensitivity-style gradients (reference ``src/models/GOKU.jl:98-130``).
mlp    numpy restatement of the LatentODE matrix-state solve (``src/models/LatentODE.jl:61-78``)
       with its continuous and discrete adjoints.
loss   numpy restatement of the ELBO reduction, reparameterised ``sample`` and Flux ``ADAMW``.
recurrent  float64 torch loops of the recurrent pattern extractor.
model  float64 torch restatement of whole GOKU_basic / LatentODE training steps over named parameters, with the
       solve as an autograd node over ``goku`` / ``mlp``.
"""
