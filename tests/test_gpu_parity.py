"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the C ABI, against the
golden vectors recorded from the reference and against the CPU oracle on seeded inputs."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, golden_cases

pytestmark = pytest.mark.gpu

Q_RTOL = 1e-3      # north_star: Q-values within 1e-3 relative in fp32
Q_ATOL_FRAC = 1e-4  # x max|Q| of the row: floor for entries near zero (10x below the 1e-3 scale)


def load(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def basin(z):
    b = float(z["basin_reward"])
    return None if b < 0 else b


def weights_dict(z):
    from oracle.mpnn import weights_from_npz
    return weights_from_npz(z)


@pytest.fixture(scope="module")
def eng():
    import eco_dqn_b200.engine as engine
    assert torch.cuda.is_available()
    return engine


def make_env(eng, z, B=None):
    gs = eng.GraphSet(z["J"][None])
    B = z["init_spins"].shape[0] if B is None else B
    env = eng.BatchedSpinSystem(gs, B, int(z["T"]), basin(z))
    env.reset(spins=z["init_spins"][:B], graph_idx=np.zeros(B, dtype=np.int32))
    return gs, env


@pytest.mark.parametrize("name", golden_cases())
def test_env_step_teacher_forced_bit_exact(eng, name):
    z = load(name)
    T, n = int(z["T"]), int(z["n"])
    gs, env = make_env(eng, z)
    B = env.B
    assert float(gs.mlr[0]) == float(z["mlr"]) and float(gs.qn[0]) == float(z["qn"]) and float(gs.lb[0]) == float(z["lb"])
    ep = env.episodes()
    assert np.array_equal(ep["score"], z["init_score"]) and np.array_equal(ep["cut"].astype(np.float64), z["init_cut"])
    k = z["obs"].shape[0]
    obs_steps = list(z["obs_steps"])
    rewards = np.zeros((B, T))
    dones = np.zeros((B, T), dtype=np.uint8)
    scores = np.zeros((B, T + 1))
    scores[:, 0] = ep["score"]
    best_scores = np.zeros((B, T + 1))
    best_scores[:, 0] = ep["best_score"]
    acts = torch.from_numpy(z["actions"]).cuda()
    for t in range(T):
        if t in obs_steps:
            got = env.observation()[:k].cpu().numpy()
            assert np.array_equal(got, z["obs"][:, obs_steps.index(t)]), (name, "obs at step", t)
        r, d = env.step(acts[:, t])
        rewards[:, t] = r.cpu().numpy()
        dones[:, t] = d.cpu().numpy()
        ep = env.episodes()
        scores[:, t + 1] = ep["score"]
        best_scores[:, t + 1] = ep["best_score"]
    if T in obs_steps:
        assert np.array_equal(env.observation()[:k].cpu().numpy(), z["obs"][:, obs_steps.index(T)])
    assert np.array_equal(rewards.view(np.uint64), z["rewards"].view(np.uint64)), "fp64 rewards must be bit-exact"
    assert np.array_equal(scores, z["scores"])
    assert np.array_equal(best_scores, z["best_scores"])
    assert np.array_equal(dones, z["dones"])
    bc, bs, st = env.results()
    assert np.array_equal(bc.cpu().numpy().astype(np.float64), z["best_cut"])
    assert np.array_equal(bs.cpu().numpy(), z["best_spins"])
    assert np.array_equal(env.spins[:, :n].cpu().numpy(), z["final_spins"])
    assert (st.cpu().numpy() == T).all()
    with pytest.raises(NotImplementedError):     # spinsystem.py:365-367
        env.step(acts[:, 0])


@pytest.mark.parametrize("impl", ["simt", "tc"])
@pytest.mark.parametrize("name", golden_cases())
def test_mpnn_q_values_and_argmax(eng, name, impl):
    from eco_dqn_b200 import _lib
    z = load(name)
    T = int(z["T"])
    gs, env = make_env(eng, z)
    w = eng.MPNNWeights(weights_dict(z))
    if impl == "tc" and w.c.packed is None:
        pytest.skip("tcgen05 path not built")
    code = _lib.MPNN_SIMT if impl == "simt" else _lib.MPNN_TCGEN05
    k = z["obs"].shape[0]
    obs_steps = list(z["obs_steps"])
    acts = torch.from_numpy(z["actions"]).cuda()
    worst = 0.0
    for t in range(T + 1):
        if t in obs_steps:
            q, a = env.q_values(w, impl=code)
            q = q[:k].cpu().numpy()
            ref = z["q"][:, obs_steps.index(t)]
            atol = Q_ATOL_FRAC * np.abs(ref).max(axis=1, keepdims=True)
            err = np.abs(q - ref) - (Q_RTOL * np.abs(ref) + atol)
            assert (err <= 0).all(), (name, t, float(np.abs(q - ref).max()))
            worst = max(worst, float((np.abs(q - ref) / (np.abs(ref) + atol)).max()))
            # argmax: lowest index among maxima, and it must be a maximiser of the reference's Q up to tolerance
            a = a[:k].cpu().numpy()
            assert np.array_equal(a, q.argmax(1))
            pick = ref[np.arange(k), a]
            assert (pick >= ref.max(1) - (Q_RTOL * np.abs(ref.max(1)) + atol[:, 0])).all()
        if t < T:
            env.step(acts[:, t])
    print("%s %s worst relative Q error %.3g" % (name, impl, worst))


@pytest.mark.parametrize("name", ["er20_g0", "er20_g3_nobasin", "ba40u_g0", "er40_g0"])
def test_free_running_rollout_against_oracle(eng, name):
    """Free-running greedy-Q rollout on the GPU; then replay the GPU's own actions through the CPU oracle:
    rewards / scores / best cuts must be bit-exact and every action must maximise the oracle's Q."""
    from oracle.rollout import rollout as cpu_rollout
    from oracle.mpnn import mpnn_forward
    z = load(name)
    T, n = int(z["T"]), int(z["n"])
    gs, env = make_env(eng, z)
    wd = weights_dict(z)
    w = eng.MPNNWeights(wd)
    ha, hr, hs = env.rollout(w, record_history=True)
    ha, hr, hs = ha.cpu().numpy(), hr.cpu().numpy(), hs.cpu().numpy()
    slack = []

    def hook(t, qs):
        qs = qs.numpy()
        picked = qs[np.arange(qs.shape[0]), ha[:, t]]
        slack.append(float(((qs.max(1) - picked) / (np.abs(qs.max(1)) + 1e-6)).max()))

    ref = cpu_rollout(z["J"].astype(np.float64), wd, z["init_spins"], T, basin(z), forced_actions=ha, q_hook=hook)
    assert np.array_equal(hr.view(np.uint64), ref["rewards"].view(np.uint64))
    assert np.array_equal(hs, ref["scores"][:, 1:])
    bc, bs, _ = env.results()
    assert np.array_equal(bc.cpu().numpy().astype(np.float64), ref["best_cut"])
    assert np.array_equal(bs.cpu().numpy(), ref["best_spins"])
    assert max(slack) <= Q_RTOL, "GPU picked an action that is not an argmax of the oracle's Q"
    # identical trajectories to the reference are expected when no near-ties occur
    same = (ha == z["actions"]).all(axis=1).mean()
    print("%s: %.0f%% of episodes follow the reference's action sequence exactly" % (name, 100 * same))
    assert bc.cpu().numpy().max() <= z["best_cut"].max() + 1e9  # (upper bound checked in known-answer test)


@pytest.mark.parametrize("n,p,B,T", [(230, 0.1, 3, 24), (300, 0.08, 2, 16)])
def test_free_running_rollout_large_graph_against_oracle(eng, n, p, B, T):
    """N > 208 (operand-tile pipeline, mpnn_large.cu) inside eco_rollout: the GPU's own action sequence replayed through
    the CPU oracle -- rewards / scores / best cuts bit-exact, every action an argmax of the oracle's Q."""
    from oracle.rollout import rollout as cpu_rollout
    from oracle.mpnn import KEYS
    from eco_dqn_b200 import _lib
    rng = np.random.default_rng(n)
    J = _random_graphs(rng, 1, n, p)
    wd = {k: (rng.standard_normal(s) * (0.3 if len(s) > 1 else 0.1)).astype(np.float32)
          for k, s in zip(KEYS, eng.STATE_DICT_SHAPES)}
    init = (2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)
    gs = eng.GraphSet(J)
    env = eng.BatchedSpinSystem(gs, B, T, 1.0 / n, mpnn_impl=_lib.MPNN_TCGEN05)
    env.reset(spins=init)
    ha, hr, hs = env.rollout(eng.MPNNWeights(wd), record_history=True)
    ha, hr, hs = ha.cpu().numpy(), hr.cpu().numpy(), hs.cpu().numpy()
    slack = []

    def hook(t, qs):
        qs = qs.numpy()
        picked = qs[np.arange(qs.shape[0]), ha[:, t]]
        slack.append(float(((qs.max(1) - picked) / (np.abs(qs.max(1)) + 1e-6)).max()))

    ref = cpu_rollout(J[0].astype(np.float64), wd, init, T, 1.0 / n, forced_actions=ha, q_hook=hook)
    assert np.array_equal(hr.view(np.uint64), ref["rewards"].view(np.uint64))
    assert np.array_equal(hs, ref["scores"][:, 1:])
    bc, bs, _ = env.results()
    assert np.array_equal(bc.cpu().numpy().astype(np.float64), ref["best_cut"])
    assert np.array_equal(bs.cpu().numpy(), ref["best_spins"])
    assert max(slack) <= Q_RTOL, "GPU picked an action that is not an argmax of the oracle's Q"


_CHUNK_SCRIPT = """
import sys, numpy as np, torch
sys.path.insert(0, %r)
import eco_dqn_b200.engine as eng
from eco_dqn_b200 import _lib
z = np.load(sys.argv[1])
gs = eng.GraphSet(z["J"])
B, n = z["spins"].shape
env = eng.BatchedSpinSystem(gs, B, 2 * n, 1.0 / n)
env.reset(spins=z["spins"], graph_idx=z["gidx"])
w = eng.MPNNWeights({k[2:]: z[k] for k in z.files if k.startswith("w_")})
q, a = env.q_values(w, impl=_lib.MPNN_TCGEN05)
np.savez(sys.argv[2], q=q.cpu().numpy(), a=a.cpu().numpy())
"""


def test_mpnn_large_graph_passes_match_single_pass(eng, tmp_path):
    """The large-graph pipeline processes episodes in passes when its planes would exceed the scratch budget
    (mpnn_large.cu: tcl_chunk); forced here to 3 episodes per pass in a child process: identical Q and actions."""
    import subprocess
    import sys
    from oracle.mpnn import KEYS
    from eco_dqn_b200 import _lib
    rng = np.random.default_rng(11)
    n, B = 300, 7
    Js = _random_graphs(rng, 2, n, 0.08)
    gidx = (np.arange(B) % 2).astype(np.int32)
    spins = (2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)
    wd = {k: (rng.standard_normal(s) * (0.3 if len(s) > 1 else 0.1)).astype(np.float32)
          for k, s in zip(KEYS, eng.STATE_DICT_SHAPES)}
    env = eng.BatchedSpinSystem(eng.GraphSet(Js), B, 2 * n, 1.0 / n)
    env.reset(spins=spins, graph_idx=gidx)
    q, a = env.q_values(eng.MPNNWeights(wd), impl=_lib.MPNN_TCGEN05)
    inp, out = str(tmp_path / "in.npz"), str(tmp_path / "out.npz")
    np.savez(inp, J=Js, spins=spins, gidx=gidx, **{"w_" + k: v for k, v in wd.items()})
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env_vars = dict(os.environ, ECO_TCL_CHUNK="3")
    subprocess.run([sys.executable, "-c", _CHUNK_SCRIPT % root, inp, out], check=True, env=env_vars, timeout=300)
    z = np.load(out)
    assert np.array_equal(z["q"], q.cpu().numpy()) and np.array_equal(z["a"], a.cpu().numpy())


@pytest.mark.parametrize("name", golden_cases())
def test_greedy_baseline_bit_exact(eng, name):
    z = load(name)
    gs, env = make_env(eng, z)
    env.rollout(policy="greedy")
    bc, bs, st = env.results()
    assert np.array_equal(bc.cpu().numpy().astype(np.float64), z["greedy_cuts"])
    assert np.array_equal(bs.cpu().numpy(), z["greedy_spins"])
    assert np.array_equal(st.cpu().numpy(), z["greedy_steps"])
    env1 = eng.BatchedSpinSystem(gs, 1, int(z["T"]), basin(z))
    env1.reset(spins=-np.ones((1, int(z["n"])), dtype=np.int8))
    env1.rollout(policy="greedy")
    bc1, bs1, _ = env1.results()
    assert float(bc1[0]) == float(z["greedy_single_cut"])
    assert np.array_equal(bs1.cpu().numpy()[0], z["greedy_single_spins"])


def _random_graphs(rng, G, n, p, pm1=True):
    out = np.zeros((G, n, n), dtype=np.int8)
    for g in range(G):
        up = np.triu((rng.random((n, n)) < p), 1)
        w = np.where(rng.random((n, n)) < 0.5, -1, 1) if pm1 else np.ones((n, n), dtype=int)
        a = (up * w).astype(np.int8)
        out[g] = a + a.T
    return out


@pytest.mark.parametrize("n,p,B,steps", [(1 + 16, 0.3, 5, 34), (16, 0.5, 3, 32), (200, 0.04, 12, 60), (333, 0.05, 4, 40),
                                         (500, 0.15, 3, 30), (1100, 0.01, 2, 20), (2000, 0.01, 2, 12)])
def test_env_random_actions_multi_graph_vs_oracle(eng, n, p, B, steps):
    """Ragged sizes (N not a multiple of 16, sub-warp / warp / block kernels), several graphs per batch."""
    from oracle.spin_env import MaxCutEnv
    rng = np.random.default_rng(n)
    G = min(B, 3)
    Js = _random_graphs(rng, G, n, p)
    gidx = (np.arange(B) * 7 % G).astype(np.int32)
    spins = (2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)
    T = 2 * n
    gs = eng.GraphSet(Js)
    env = eng.BatchedSpinSystem(gs, B, T, 1.0 / n)
    env.reset(spins=spins, graph_idx=gidx)
    cpu = [MaxCutEnv(Js[gidx[b]].astype(np.float64), T, 1.0 / n) for b in range(B)]
    obs = [e.reset(spins[b]) for b, e in enumerate(cpu)]
    for t in range(steps):
        got = env.observation().cpu().numpy()
        want = np.stack([o[:7] for o in obs]).astype(np.float32)
        assert np.array_equal(got, want), ("obs", t)
        # mix of random moves, revisits (to exercise the visited set) and greedy moves
        if t % 5 == 4:
            a = np.array([int(np.argmax(e.spins * (e.J @ e.spins))) for e in cpu])
        elif t % 7 == 6:
            a = prev
        else:
            a = rng.integers(0, n, size=B)
        prev = a
        r, d = env.step(torch.from_numpy(a.astype(np.int32)))
        out = [e.step(int(x)) for e, x in zip(cpu, a)]
        obs = [o[0] for o in out]
        assert np.array_equal(r.cpu().numpy().view(np.uint64), np.array([o[1] for o in out], dtype=np.float64).view(np.uint64))
    ep = env.episodes()
    assert np.array_equal(ep["score"], np.array([e.score for e in cpu]))
    assert np.array_equal(ep["best_cut"].astype(np.float64), np.array([e.best_solution for e in cpu]))
    _, bs, _ = env.results()
    assert np.array_equal(bs.cpu().numpy(), np.stack([e.best_spins for e in cpu]).astype(np.int8))


@pytest.mark.parametrize("n,variant", [(129, "fast"), (200, "fast"), (241, "fast"), (256, "fast"),
                                       (200, "weights"), (232, "long")])
def test_env_step_staged_ring_matches_subwarp_kernel(eng, n, variant):
    """B >= 4096 with caller-supplied actions runs env_step_ring_kernel (persistent warps, async-copy ring); smaller batches
    run the sub-warp kernel that the oracle tests pin.  Same episodes, same actions (out-of-range ones included): every
    state array, observation, reward and done flag must be identical.  "fast": the rollout configuration (+-1 couplings,
    T + 1 <= 1024: the FAST instantiation); "weights": couplings in -3 .. 3 and "long": T = 1100, both through the general
    instantiation."""
    rng = np.random.default_rng(1000 + n)
    B, G, T, steps = 4096 + 37, 5, 24, 24       # T small: episodes finish inside the test, done episodes stay untouched
    if variant == "long":
        T = 1100
    Js = _random_graphs(rng, G, n, 0.06)
    if variant == "weights":
        mag = np.triu(rng.integers(1, 4, size=Js.shape), 1).astype(np.int8)
        Js = Js * (mag + mag.transpose(0, 2, 1))
    gidx = rng.integers(0, G, size=B).astype(np.int32)
    spins = (2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)
    gs = eng.GraphSet(Js)
    big = eng.BatchedSpinSystem(gs, B, T, 1.0 / n)
    big.reset(spins=spins, graph_idx=gidx)
    parts = []
    for lo in range(0, B, 2048):
        hi = min(B, lo + 2048)
        e = eng.BatchedSpinSystem(gs, hi - lo, T, 1.0 / n)
        e.reset(spins=spins[lo:hi], graph_idx=gidx[lo:hi])
        parts.append((lo, hi, e))
    for t in range(steps):
        a = rng.integers(0, n, size=B).astype(np.int32)
        if t % 6 == 5:
            a[::3] = prev[::3]                   # revisits: exercise the visited-set probe
        if t == 7:
            a[5] = -1; a[11] = n                 # invalid actions are ignored (episode left untouched, done reported)
        prev = a
        r, d = big.step(torch.from_numpy(a))
        r, d = r.cpu().numpy(), d.cpu().numpy()
        for lo, hi, e in parts:
            rp, dp = e.step(torch.from_numpy(a[lo:hi]))
            assert np.array_equal(r[lo:hi].view(np.uint64), rp.cpu().numpy().view(np.uint64)), ("reward", t)
            assert np.array_equal(d[lo:hi], dp.cpu().numpy()), ("done", t)
        if t % 5 == 0 or t == steps - 1:
            ob = big.observation().cpu().numpy()
            epb = big.episodes()
            for lo, hi, e in parts:
                assert np.array_equal(ob[lo:hi], e.observation().cpu().numpy()), ("obs", t)
                assert epb[lo:hi].tobytes() == e.episodes().tobytes(), ("episode block", t)
    bc, bs, st = big.results()
    for lo, hi, e in parts:
        bcp, bsp, stp = e.results()
        assert torch.equal(bc[lo:hi], bcp) and torch.equal(bs[lo:hi], bsp) and torch.equal(st[lo:hi], stp)


@pytest.mark.parametrize("n,p", [(24, 0.3), (200, 0.15), (500, 0.05)])
def test_mpnn_simt_random_weights_multi_graph_vs_oracle(eng, n, p):
    from oracle.mpnn import mpnn_forward, KEYS
    from eco_dqn_b200 import _lib
    rng = np.random.default_rng(n + 1)
    B, G = 6, 3
    Js = _random_graphs(rng, G, n, p)
    gidx = (np.arange(B) % G).astype(np.int32)
    shapes = eng.STATE_DICT_SHAPES
    wd = {k: (rng.standard_normal(s) * (0.3 if len(s) > 1 else 0.1)).astype(np.float32) for k, s in zip(KEYS, shapes)}
    gs = eng.GraphSet(Js)
    env = eng.BatchedSpinSystem(gs, B, 2 * n, 1.0 / n)
    env.reset(spins=(2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8), graph_idx=gidx)
    for t in range(5):
        env.step(torch.from_numpy(rng.integers(0, n, size=B).astype(np.int32)))
    w = eng.MPNNWeights(wd)
    q, a = env.q_values(w, impl=_lib.MPNN_SIMT)
    obs7 = env.observation().cpu().numpy()
    full = np.concatenate([obs7, Js[gidx].astype(np.float32)], axis=1)
    ref = mpnn_forward(wd, full).numpy()      # batch-wide norm.max() == max degree over the set here
    deg_max_batch = max((Js[g] != 0).sum(1).max() for g in gidx)
    assert deg_max_batch == gs.max_degree
    q = q.cpu().numpy()
    assert np.allclose(q, ref, rtol=Q_RTOL, atol=Q_ATOL_FRAC * np.abs(ref).max())
    assert np.array_equal(a.cpu().numpy(), q.argmax(1))


@pytest.mark.parametrize("n,B", [(5, 40), (17, 29), (20, 13), (33, 10), (48, 9), (64, 7), (90, 5), (96, 2)])
@pytest.mark.parametrize("norm_max", [None, -1.0])
def test_mpnn_tc_packed_small_graphs_vs_oracle(eng, n, B, norm_max):
    """Small graphs are processed K = 192 / NP at a time as one block-diagonal graph (packed mode): several DIFFERENT
    graphs per pack, ragged N, a partial last pack, per-episode graph-level observations; norm_max < 0 = the per-graph
    degree normalisation the single-env facade uses."""
    from oracle.mpnn import mpnn_forward, KEYS
    from eco_dqn_b200 import _lib
    rng = np.random.default_rng(7 * n + B)
    G = min(B, 5)
    Js = _random_graphs(rng, G, n, 0.8, pm1=False) if n < 10 else _random_graphs(rng, G, n, 0.3 if n < 40 else 0.1)
    gidx = rng.integers(0, G, size=B).astype(np.int32)
    shapes = eng.STATE_DICT_SHAPES
    wd = {k: (rng.standard_normal(s) * (0.3 if len(s) > 1 else 0.1)).astype(np.float32) for k, s in zip(KEYS, shapes)}
    gs = eng.GraphSet(Js)
    env = eng.BatchedSpinSystem(gs, B, 2 * n, 1.0 / n)
    env.reset(spins=(2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8), graph_idx=gidx)
    for t in range(1 + n // 4):                  # different step counts of progress per episode are not possible; vary spins
        env.step(torch.from_numpy(rng.integers(0, n, size=B).astype(np.int32)))
    w = eng.MPNNWeights(wd)
    if norm_max is None:                         # the reference's norm.max() over the batch it is given (mpnn.py:102)
        norm_max = float(max((Js[g] != 0).sum(1).max() for g in gidx))
        per_graph = False
    else:
        per_graph = True
    q, a = env.q_values(w, impl=_lib.MPNN_TCGEN05, norm_max=norm_max)
    q2, a2 = env.q_values(w, impl=_lib.MPNN_TCGEN05, norm_max=norm_max)
    assert torch.equal(q, q2) and torch.equal(a, a2)          # run-to-run deterministic
    q, a = q.cpu().numpy(), a.cpu().numpy()
    obs7 = env.observation().cpu().numpy()
    full = np.concatenate([obs7, Js[gidx].astype(np.float32)], axis=1)
    if not per_graph:
        ref = mpnn_forward(wd, full).numpy()
    else:
        ref = np.stack([mpnn_forward(wd, full[b:b + 1]).numpy().reshape(-1) for b in range(B)])   # per-episode norm.max()
    assert np.allclose(q, ref, rtol=Q_RTOL, atol=Q_ATOL_FRAC * np.abs(ref).max())
    assert np.array_equal(a, q.argmax(1))


@pytest.mark.parametrize("n,B", [(20, 148 * 6 * 2 + 77), (40, 148 * 4 * 3 + 5)])
def test_mpnn_tc_packed_many_packs_per_cta(eng, n, B):
    """More packs than CTAs: every CTA works through several packs, so all but its last pack are read out by the tail warp
    beside the next pack's stages (the last one by all epilogue warps), and the operand-image blocks of the next pack are
    fetched by the contraction issuer.  Q against the oracle; and an episode's Q bits must not depend on where in the launch
    it was evaluated: the first episodes again as a batch of their own (one pack per CTA, all-worker readout)."""
    from oracle.mpnn import mpnn_forward, KEYS
    from eco_dqn_b200 import _lib
    rng = np.random.default_rng(31 * n + B)
    G = 64
    Js = _random_graphs(rng, G, n, 0.3 if n < 40 else 0.15)
    gidx = rng.integers(0, G, size=B).astype(np.int32)
    spins = (2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)
    wd = {k: (rng.standard_normal(s) * (0.3 if len(s) > 1 else 0.1)).astype(np.float32)
          for k, s in zip(KEYS, eng.STATE_DICT_SHAPES)}
    w = eng.MPNNWeights(wd)
    gs = eng.GraphSet(Js)
    acts = [rng.integers(0, n, size=B).astype(np.int32) for _ in range(3)]

    def run(count):
        env = eng.BatchedSpinSystem(gs, count, 2 * n, 1.0 / n)
        env.reset(spins=spins[:count], graph_idx=gidx[:count])
        for a in acts:
            env.step(torch.from_numpy(a[:count].copy()))
        q, a = env.q_values(w, impl=_lib.MPNN_TCGEN05, norm_max=-1.0)
        return env, q.clone(), a.clone()

    env, q, a = run(B)
    q2, a2 = env.q_values(w, impl=_lib.MPNN_TCGEN05, norm_max=-1.0)
    assert torch.equal(q, q2) and torch.equal(a, a2)                      # run-to-run deterministic
    small = 37
    _, qs, a_s = run(small)
    assert torch.equal(q[:small], qs) and torch.equal(a[:small], a_s)     # same bits wherever the episode sits in the launch
    obs7 = env.observation().cpu().numpy()
    q, a = q.cpu().numpy(), a.cpu().numpy()
    assert np.array_equal(a, q.argmax(1))
    check = np.concatenate([np.arange(0, 64), rng.choice(B, size=192, replace=False), np.arange(B - 64, B)])
    for b in check:                                                        # per-episode norm.max() (norm_max < 0)
        full = np.concatenate([obs7[b:b + 1], Js[gidx[b]][None].astype(np.float32)], axis=1)
        ref = mpnn_forward(wd, full).numpy().reshape(-1)
        assert np.allclose(q[b], ref, rtol=Q_RTOL, atol=Q_ATOL_FRAC * np.abs(ref).max()), b
    q_si, _ = env.q_values(w, impl=_lib.MPNN_SIMT, norm_max=-1.0)
    q_si = q_si.cpu().numpy()
    assert np.all(np.abs(q - q_si) <= Q_RTOL * np.abs(q_si) + Q_ATOL_FRAC * np.abs(q_si).max(1, keepdims=True))


def test_full_size_invariants_ba200(eng):
    """BASELINE config 2 size (B=4096, N=200): size-independent properties after a greedy + random walk."""
    gsets = np.load(os.path.join(GOLDEN, "graphsets.npz"))
    Js = gsets["ba200"]
    B, n, T = 4096, 200, 400
    rng = np.random.default_rng(0)
    gs = eng.GraphSet(Js)
    env = eng.BatchedSpinSystem(gs, B, T, 1.0 / n)
    spins0 = torch.from_numpy((2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)).cuda()
    env.reset(spins=spins0)
    gen = torch.Generator(device="cuda").manual_seed(1)
    for t in range(60):
        env.step(torch.randint(0, n, (B,), generator=gen, device="cuda", dtype=torch.int32))
    for t in range(40):
        env.greedy_step()
    ep = env.episodes()
    s = env.spins[:, :n].float()
    J = gs.J[:, :n, :n].float()[env.graph_idx.long()]
    h = torch.bmm(J, s.unsqueeze(-1)).squeeze(-1)
    assert torch.equal(h, env.hfield[:, :n].float())
    cut = 0.25 * (J.sum((1, 2)) - (s * h).sum(1))
    assert np.array_equal(cut.cpu().numpy(), ep["cut"].astype(np.float32))
    bc, bs, st = env.results()
    bsf = bs.float()
    bcut = 0.25 * (J.sum((1, 2)) - (bsf * torch.bmm(J, bsf.unsqueeze(-1)).squeeze(-1)).sum(1))
    assert torch.equal(bcut, bc.float())
    assert np.array_equal((bs != env.spins[:, :n]).sum(1).cpu().numpy(), ep["dist"])
    assert (ep["best_score"] >= ep["score"]).all() and (ep["step"] <= 100).all()
    opt = gsets["ba200_opt"][(np.arange(B) % Js.shape[0])]
    assert (bc.cpu().numpy() <= opt).all()          # best-known cuts are upper bounds (README.md:82)


@pytest.mark.parametrize("n,p,B,G,steps", [(500, 0.15, 4096, 8, 24), (2000, 0.01, 192, 3, 10)])
def test_full_size_invariants_large_graphs(eng, n, p, B, G, steps):
    """BASELINE configs 3 / 4 sizes (ER-500 with 4096 episodes per GPU; GSet-shaped 2000-vertex +-1 graphs): a network
    rollout segment (CUDA-core MPNN: N > 208) followed by greedy steps, then size-independent properties -- local fields
    and cut recomputed from the spins, best spins reproduce the best cut, Hamming distance, argmax consistency."""
    rng = np.random.default_rng(n)
    Js = _random_graphs(rng, G, n, p)
    gs = eng.GraphSet(Js)
    T = 2 * n
    env = eng.BatchedSpinSystem(gs, B, T, 1.0 / n)
    env.reset(spins=torch.from_numpy((2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)).cuda())
    w = eng.MPNNWeights(weights_dict(load("er200_g0")))
    ha, hr, hs = env.rollout(w, n_steps=steps, record_history=True)
    q, a = env.q_values(w)
    assert torch.equal(a.long(), q.argmax(1))                       # fused argmax == argmax of the written Q (lowest index)
    assert bool(torch.isfinite(q).all())
    for t in range(6):
        env.greedy_step()
    ep = env.episodes()
    assert (ep["step"] <= steps + 6).all() and (ep["step"] >= steps).all()
    sel = torch.arange(0, B, max(1, B // 64), device="cuda")        # a sample of episodes (N^2 work on the host side)
    s = env.spins[sel, :n].float()
    J = gs.J[:, :n, :n].float()[env.graph_idx[sel].long()]
    h = torch.bmm(J, s.unsqueeze(-1)).squeeze(-1)
    assert torch.equal(h, env.hfield[sel, :n].float())
    cut = 0.25 * (J.sum((1, 2)) - (s * h).sum(1))
    assert np.array_equal(cut.cpu().numpy(), ep["cut"][sel.cpu().numpy()].astype(np.float32))
    bc, bs, st = env.results()
    bsf = bs[sel].float()
    bcut = 0.25 * (J.sum((1, 2)) - (bsf * torch.bmm(J, bsf.unsqueeze(-1)).squeeze(-1)).sum(1))
    assert torch.equal(bcut, bc[sel].float())
    assert np.array_equal((bs != env.spins[:, :n]).sum(1).cpu().numpy(), ep["dist"])
    assert (ep["best_score"] >= ep["score"]).all()
    # the recorded scores are consistent with the recorded rewards' sign structure: best score = running max
    hs = hs.cpu().numpy()[:, :steps]
    assert np.all(ep["best_score"] >= hs.max(1))


def test_host_session_matches_engine(eng):
    z = load("er20_g0")
    from eco_dqn_b200 import _lib
    T, n = int(z["T"]), int(z["n"])
    B = z["init_spins"].shape[0]
    wd = weights_dict(z)
    sess = eng.HostSession(1, n, B, T, basin(z), wd, impl=_lib.MPNN_SIMT)
    best_cut = np.zeros(B, dtype=np.int32)
    best_spins = np.zeros((B, n), dtype=np.int8)
    sess.rollout(np.ascontiguousarray(z["J"][None]), np.zeros(B, dtype=np.int32), np.ascontiguousarray(z["init_spins"]),
                 best_cut, best_spins)
    gs, env = make_env(eng, z)
    env.rollout(eng.MPNNWeights(wd), impl=_lib.MPNN_SIMT)
    bc, bs, _ = env.results()
    assert np.array_equal(best_cut, bc.cpu().numpy()) and np.array_equal(best_spins, bs.cpu().numpy())
    sess.close()


def test_host_session_large_graph_matches_engine(eng):
    """Host-buffer session on a graph with N > 208 (AUTO -> the operand-tile pipeline) against the engine."""
    from oracle.mpnn import KEYS
    from eco_dqn_b200 import _lib
    rng = np.random.default_rng(5)
    n, B, T = 230, 4, 12
    J = _random_graphs(rng, 2, n, 0.1)
    gidx = np.array([0, 1, 1, 0], dtype=np.int32)
    init = (2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)
    wd = {k: (rng.standard_normal(s) * (0.3 if len(s) > 1 else 0.1)).astype(np.float32)
          for k, s in zip(KEYS, eng.STATE_DICT_SHAPES)}
    sess = eng.HostSession(2, n, B, T, 1.0 / n, wd, impl=_lib.MPNN_AUTO)
    best_cut = np.zeros(B, dtype=np.int32)
    best_spins = np.zeros((B, n), dtype=np.int8)
    sess.rollout(np.ascontiguousarray(J), gidx, init, best_cut, best_spins)
    env = eng.BatchedSpinSystem(eng.GraphSet(J), B, T, 1.0 / n)
    env.reset(spins=init, graph_idx=gidx)
    env.rollout(eng.MPNNWeights(wd))
    bc, bs, _ = env.results()
    assert np.array_equal(best_cut, bc.cpu().numpy()) and np.array_equal(best_spins, bs.cpu().numpy())
    sess.close()


def test_error_behaviour(eng):
    z = load("er20_g0")
    gs, env = make_env(eng, z)
    with pytest.raises(Exception):        # spinsystem.py:604-606
        env.reset(spins=np.zeros((env.B, env.N), dtype=np.int8))
    with pytest.raises(NotImplementedError):   # real-valued couplings are outside the accelerated path
        eng.GraphSet(np.array([[0, 0.5], [0.5, 0]])[None])
    with pytest.raises(ValueError):        # empty graph: the reference recurses forever (spinsystem.py:209-211)
        eng.GraphSet(np.zeros((1, 8, 8)))
    with pytest.raises(ValueError):
        eng.GraphSet(np.triu(np.ones((1, 8, 8)), 1))   # not symmetric


def test_mpnn_tc_is_run_to_run_deterministic(eng):
    """Chunks are handed out dynamically to the two warp groups; results must not depend on the hand-out."""
    from eco_dqn_b200 import _lib
    gsets = np.load(os.path.join(GOLDEN, "graphsets.npz"))
    z = load("ba200_g0")
    B, n = 2048, 200
    rng = np.random.default_rng(3)
    gs = eng.GraphSet(gsets["ba200"])
    env = eng.BatchedSpinSystem(gs, B, 400, 1.0 / n)
    env.reset(spins=(2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8))
    w = eng.MPNNWeights(weights_dict(z))
    if w.c.packed is None:
        pytest.skip("tcgen05 path not built")
    for t in range(3):
        q1, a1 = env.q_values(w, impl=_lib.MPNN_TCGEN05)
        q1, a1 = q1.clone(), a1.clone()
        for rep in range(3):
            q2, a2 = env.q_values(w, impl=_lib.MPNN_TCGEN05)
            assert torch.equal(q1, q2) and torch.equal(a1, a2)
        qs, _ = env.q_values(w, impl=_lib.MPNN_SIMT)
        assert torch.allclose(q1, qs, rtol=Q_RTOL, atol=Q_ATOL_FRAC * float(qs.abs().max()))
        env.step(a1)


# ---------------------------------------------------------------------------------------------------------------
# S2V-DQN configuration (SURVEY.md section 8(f)3): irreversible spins, spin-only observation, dense reward
# ---------------------------------------------------------------------------------------------------------------
from conftest import s2v_cases            # noqa: E402


@pytest.mark.parametrize("name", s2v_cases())
def test_s2v_teacher_forced_and_q_values(eng, name):
    z = load(name)
    n, T = int(z["n"]), int(z["T"])
    gs = eng.GraphSet(z["J"][None])
    w = eng.MPNNWeights(weights_dict(z))
    assert w.n_obs_in == 1
    env = eng.BatchedSpinSystem(gs, 1, T, None, reversible_spins=False, dense_reward=True)
    env.reset()
    assert np.array_equal(env.spins[0, :n].cpu().numpy(), -np.ones(n, dtype=np.int8))
    assert env.episodes()["score"][0] == float(z["init_score"])
    for t, a in enumerate(z["actions"]):
        q, act = env.q_values(w, norm_max=-1.0)              # one episode: norm.max() is this graph's max degree
        q = q.cpu().numpy()[0]
        assert np.allclose(q, z["q"][t], rtol=Q_RTOL, atol=Q_ATOL_FRAC * np.abs(z["q"][t]).max()), ("q", t)
        assert int(act[0]) == int(a), ("masked argmax", t)
        r, d = env.step(torch.tensor([int(a)], dtype=torch.int32))
        r = r.cpu().numpy()
        assert r[0] == z["rewards"][t] and np.signbit(r[0]) == np.signbit(z["rewards"][t]), ("reward", t)
        assert int(d[0]) == int(z["dones"][t]) and env.episodes()["score"][0] == z["scores"][t + 1]
        assert np.array_equal(env.spins[0, :n].cpu().numpy(), z["spins"][t + 1])
    bc, bs, st = env.results()
    assert float(bc[0]) == float(z["best_cut"]) and np.array_equal(bs[0].cpu().numpy(), z["best_spins"])


@pytest.mark.parametrize("name", s2v_cases())
def test_s2v_device_rollout_and_greedy(eng, name):
    z = load(name)
    n, T = int(z["n"]), int(z["T"])
    gs = eng.GraphSet(z["J"][None])
    w = eng.MPNNWeights(weights_dict(z))
    env = eng.BatchedSpinSystem(gs, 3, T, None, reversible_spins=False, dense_reward=True)   # 3 identical episodes
    env.reset(graph_idx=np.zeros(3, dtype=np.int32))
    ha, hr, hs = env.rollout(w, record_history=True)
    ha, hr = ha.cpu().numpy(), hr.cpu().numpy()
    k = len(z["actions"])
    for b in range(3):
        assert np.array_equal(ha[b, :k], z["actions"]) and np.array_equal(hr[b, :k], z["rewards"])
    bc, bs, st = env.results()
    assert float(bc[0]) == float(z["best_cut"]) and int(st[0]) == k
    g = eng.BatchedSpinSystem(gs, 2, T, None, reversible_spins=False, dense_reward=True)
    g.reset(graph_idx=np.zeros(2, dtype=np.int32))
    g.rollout(policy="greedy")
    bc, bs, st = g.results()
    assert float(bc[1]) == float(z["greedy_cut"]) and np.array_equal(bs[1].cpu().numpy(), z["greedy_spins"])
    assert int(st[1]) == int(z["greedy_steps"])


def test_s2v_rollout_large_graph_against_oracle(eng):
    """S2V-DQN configuration on a graph with N > 208: the operand-tile pipeline feeds the masked argmax inside
    eco_rollout.  The GPU's action sequence is replayed through the oracle: rewards (with their sign bits), scores and
    done flags bit-exact, every action a masked argmax of the oracle's Q."""
    from oracle.rollout import rollout_s2v
    from oracle.mpnn import KEYS
    rng = np.random.default_rng(23)
    n, T = 240, 40
    J = _random_graphs(rng, 1, n, 0.08)
    wd = {k: (rng.standard_normal(s) * (0.3 if len(s) > 1 else 0.1)).astype(np.float32)
          for k, s in zip(KEYS, eng.STATE_DICT_SHAPES)}
    wd[KEYS[0]] = wd[KEYS[0]][:, :1].copy()                 # n_obs_in = 1 (networks/s2v): W_init [64, 1], W_e [63, 2]
    wd[KEYS[1]] = wd[KEYS[1]][:, :2].copy()
    w = eng.MPNNWeights(wd)
    assert w.n_obs_in == 1
    env = eng.BatchedSpinSystem(eng.GraphSet(J), 2, T, None, reversible_spins=False, dense_reward=True)
    env.reset(graph_idx=np.zeros(2, dtype=np.int32))
    ha, hr, hs = env.rollout(w, record_history=True, norm_max=-1.0)
    ha, hr, hs = ha.cpu().numpy(), hr.cpu().numpy(), hs.cpu().numpy()
    assert np.array_equal(ha[0], ha[1]) and len(set(ha[0].tolist())) == T          # irreversible: T distinct vertices
    slack = []

    def hook(t, qs):
        q = qs.numpy().reshape(-1).copy()
        q[np.array(sorted(set(ha[0, :t].tolist())), dtype=np.int64)] = -np.inf
        slack.append(float((q.max() - q[ha[0, t]]) / (abs(q.max()) + 1e-6)))

    ref = rollout_s2v(J[0].astype(np.float64), wd, T, forced_actions=ha[0], q_hook=hook)
    k = len(ref["actions"])
    assert k == T
    assert np.array_equal(hr[0, :k].view(np.uint64), ref["rewards"].view(np.uint64))
    assert np.array_equal(hs[0, :k], ref["scores"][1:])
    bc, bs, st = env.results()
    assert float(bc[0]) == ref["best_cut"] and np.array_equal(bs[0].cpu().numpy(), ref["best_spins"])
    assert max(slack) <= Q_RTOL, "GPU picked an action that is not a masked argmax of the oracle's Q"


# ---------------------------------------------------------------------------------------------------------------
# OptimisationTarget.MIN_CUT (SURVEY.md section 8(f)3)
# ---------------------------------------------------------------------------------------------------------------
from conftest import mincut_cases            # noqa: E402


@pytest.mark.parametrize("name", mincut_cases())
def test_mincut_env_and_rollout_bit_exact(eng, name):
    z = load(name)
    T, n = int(z["T"]), int(z["n"])
    gs = eng.GraphSet(z["J"][None], min_cut=True)
    assert float(gs.mlr[0]) == float(z["mlr"]) and float(gs.qn[0]) == float(z["qn"]) and float(gs.lb[0]) == float(z["lb"])
    B = z["init_spins"].shape[0]
    env = eng.BatchedSpinSystem(gs, B, T, basin(z))
    env.reset(spins=z["init_spins"], graph_idx=np.zeros(B, dtype=np.int32))
    ep = env.episodes()
    assert np.array_equal(ep["score"], z["init_score"]) and np.array_equal(ep["cut"].astype(np.float64), z["init_cut"])
    k = z["obs"].shape[0]
    obs_steps = list(z["obs_steps"])
    w = eng.MPNNWeights(weights_dict(z))
    for t in range(T):
        if t in obs_steps:
            got = env.observation().cpu().numpy()[:k]
            assert np.array_equal(got, z["obs"][:, obs_steps.index(t)]), ("obs", t)
            q, _ = env.q_values(w)
            ref = z["q"][:, obs_steps.index(t)]
            assert np.allclose(q.cpu().numpy()[:k], ref, rtol=Q_RTOL, atol=Q_ATOL_FRAC * np.abs(ref).max())
        r, d = env.step(torch.from_numpy(z["actions"][:, t].copy()))
        assert np.array_equal(r.cpu().numpy().view(np.uint64), z["rewards"][:, t].view(np.uint64)), ("reward", t)
        assert np.array_equal(env.episodes()["score"], z["scores"][:, t + 1])
    bc, bs, _ = env.results()
    assert np.array_equal(bc.cpu().numpy().astype(np.float64), z["best_cut"])
    assert np.array_equal(bs.cpu().numpy(), z["best_spins"])
    # free-running network rollout and the greedy baselines
    env.reset(spins=z["init_spins"], graph_idx=np.zeros(B, dtype=np.int32))
    ha, hr, hs = env.rollout(w, record_history=True)
    assert np.array_equal(ha.cpu().numpy(), z["actions"])
    env.reset(spins=z["init_spins"], graph_idx=np.zeros(B, dtype=np.int32))
    env.rollout(policy="greedy")
    gc, gsp, gst = env.results()
    assert np.array_equal(gc.cpu().numpy().astype(np.float64), z["greedy_cuts"])
    assert np.array_equal(gsp.cpu().numpy(), z["greedy_spins"]) and np.array_equal(gst.cpu().numpy(), z["greedy_steps"])


# ---------------------------------------------------------------------------------------------------------------
# tensor-core neighbour aggregation for graphs beyond the resident kernel (eco_graph_aggregate, mpnn_tcl.cu)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,p,B", [(20, 0.3, 3), (200, 0.1, 5), (333, 0.1, 4), (500, 0.15, 6), (1100, 0.02, 3), (2000, 0.01, 2)])
@pytest.mark.parametrize("use_abs", [0, 1])
def test_graph_aggregate_matches_fp64_product(eng, n, p, B, use_abs):
    import ctypes as C
    from eco_dqn_b200 import _lib
    rng = np.random.default_rng(n + use_abs)
    G = 2
    Js = _random_graphs(rng, G, n, p)
    gs = eng.GraphSet(Js)
    gidx = torch.from_numpy((np.arange(B) % G).astype(np.int32)).cuda()
    x = torch.from_numpy(rng.standard_normal((B, n, 64)).astype(np.float32) * 3.0).cuda()
    out = torch.full((B, n, 64), float("nan"), dtype=torch.float32, device="cuda")
    eng.check(_lib.lib().eco_graph_aggregate(C.byref(gs.c), B, C.c_void_p(gidx.data_ptr()), C.c_void_p(x.data_ptr()),
                                             use_abs, 0.5, C.c_void_p(out.data_ptr()),
                                             C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    Jd = torch.from_numpy(Js.astype(np.float64)).cuda()[gidx.long()]
    if use_abs:
        Jd = Jd.abs()
    deg = (Jd != 0).sum(1).clamp(min=1).double()                       # [B, n] (symmetric)
    ref = 0.5 * torch.einsum("bji,bjf->bif", Jd, x.double()) / deg.unsqueeze(-1)
    err = (out.double() - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert np.isfinite(err) and err <= 2e-5 * scale, (err, scale)      # bf16 hi+lo: 16 mantissa bits per term, fp32 accumulate


@pytest.mark.parametrize("n,p,B", [(209, 0.1, 5), (333, 0.08, 4), (500, 0.15, 6), (1100, 0.02, 3), (2000, 0.01, 2),
                                   (257, 0.1, 1), (2048, 0.005, 1), (500, 0.15, 333)])
@pytest.mark.parametrize("norm_max", [None, -1.0])
def test_mpnn_large_graph_tensor_path_vs_oracle_and_simt(eng, n, p, B, norm_max):
    """N > 208: the operand-tile pipeline (mpnn_large.cu: N x N products and per-vertex linears on the tensor cores),
    against the oracle (Q tolerance) and against the all-CUDA-core kernel."""
    from oracle.mpnn import mpnn_forward, KEYS
    from eco_dqn_b200 import _lib
    rng = np.random.default_rng(3 * n + B)
    G = min(2, B)             # norm_max=None: the set-wide max degree is the batch's max only if every graph is used
    Js = _random_graphs(rng, G, n, p)
    gidx = (np.arange(B) % G).astype(np.int32)
    wd = {k: (rng.standard_normal(s) * (0.3 if len(s) > 1 else 0.1)).astype(np.float32)
          for k, s in zip(KEYS, eng.STATE_DICT_SHAPES)}
    gs = eng.GraphSet(Js)
    env = eng.BatchedSpinSystem(gs, B, 2 * n, 1.0 / n)
    env.reset(spins=(2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8), graph_idx=gidx)
    for t in range(4):
        env.step(torch.from_numpy(rng.integers(0, n, size=B).astype(np.int32)))
    w = eng.MPNNWeights(wd)
    q_tc, a_tc = env.q_values(w, impl=_lib.MPNN_TCGEN05, norm_max=norm_max)
    q_tc, a_tc = q_tc.cpu().numpy().copy(), a_tc.cpu().numpy().copy()
    q_si, a_si = env.q_values(w, impl=_lib.MPNN_SIMT, norm_max=norm_max)
    q_si = q_si.cpu().numpy()
    assert np.allclose(q_tc, q_si, rtol=Q_RTOL, atol=Q_ATOL_FRAC * np.abs(q_si).max())
    assert np.array_equal(a_tc, q_tc.argmax(1))
    q_again, a_again = env.q_values(w, impl=_lib.MPNN_TCGEN05, norm_max=norm_max)
    assert np.array_equal(q_again.cpu().numpy(), q_tc) and np.array_equal(a_again.cpu().numpy(), a_tc)   # run-to-run identical
    if n <= 500 and B <= 8:                                       # the dense oracle needs B * N^2 * 63 floats
        obs7 = env.observation().cpu().numpy()
        full = np.concatenate([obs7, Js[gidx].astype(np.float32)], axis=1)
        if norm_max is None:
            ref = mpnn_forward(wd, full).numpy()
        else:
            ref = np.stack([mpnn_forward(wd, full[b:b + 1]).numpy().reshape(-1) for b in range(B)])
        assert np.allclose(q_tc, ref, rtol=Q_RTOL, atol=Q_ATOL_FRAC * np.abs(ref).max())
