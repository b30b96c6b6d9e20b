"""CPU oracle for the ECO-DQN Max-Cut rollout hot path.

TEST INFRASTRUCTURE ONLY.  This package is a CPU restatement of the reference's algorithm
(BetterBelle/eco-dqn) for the one hot path this repository accelerates.  It may be imported by
`tests/`, by `__graft_entry__.smoke()` and by `bench.py`'s `cpu_baseline` / `--impl reference`
legs, and by nothing else: the product (`eco-dqn_b200/`) never imports it and has no CPU fallback.

Parity status: PINNED.  The reference has no test suite of its own (SURVEY.md section 4), so the
oracle is pinned against outputs of the unmodified reference run in the build container:
`tests/golden/make_golden.py` drives the reference's `make` / `SpinSystemBase` / `MPNN` /
`test_network` with fixed seeds and commits the trajectories (init spins, actions, fp64 rewards and
scores, observation rows, Q-values, best cuts, greedy baselines) under `tests/golden/*.npz`;
`tests/test_oracle_golden.py` replays them through this package bit-exactly (Q-values to 1e-5).

Modules
  spin_env.py  restates src/envs/spinsystem.py + score_solver.py (MaximumCutUnbiasedScorer) +
               utils.py (calculate_cut, calculate_cut_changes, HistoryBuffer)
  mpnn.py      restates src/networks/mpnn.py (forward only, fp32, as written: dense [B,N,N,63] edge stage)
  mpnn64.py    the same forward in float64 over a CSR graph, explicit degrees and divisor, differentiable
               (the reference the kernels' precision tests compare with)
  rollout.py   restates experiments/utils.py::__test_network_batched (greedy-Q loop, Greedy baseline)
"""
