"""GPU tests of CSR graph sets (SparseGraphSet): the O(degree) environment step, the gather MPNN, the rollout, the Greedy
baseline and the drop-in routing -- bit for bit against the dense int8 path for N <= 2048, against the CPU oracle beyond."""
import os

import numpy as np
import pytest
import scipy.sparse as sps
import torch

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

Q_RTOL = 1e-3
Q_ATOL_FRAC = 1e-4


@pytest.fixture(scope="module")
def eng():
    import eco_dqn_b200.engine as engine
    assert torch.cuda.is_available()
    return engine


@pytest.fixture(scope="module")
def wd():
    from oracle.mpnn import weights_from_npz
    return weights_from_npz(np.load(os.path.join(GOLDEN, "er20_g0.npz")))


@pytest.fixture
def sparse_oracle(monkeypatch):
    """oracle.spin_env with its two O(N^2) kernels -- flip_gains (J @ s) and cut_value (outer product) -- evaluated on a CSR
    copy of the same fp64 matrix, and observation() without the N x N adjacency rows.  Integer couplings: every sum is exact
    in fp64 in any order, so the results are the dense oracle's bit for bit."""
    import oracle.spin_env as se
    cache = {}

    def csr(J):
        hit = cache.get(id(J))
        if hit is None or hit[0] is not J:
            hit = cache[id(J)] = (J, sps.csr_matrix(J))
        return hit[1]

    monkeypatch.setattr(se, "flip_gains", lambda s, J: s * (csr(J) @ s))
    monkeypatch.setattr(se, "cut_value", lambda s, J: (1 / 4) * (csr(J).sum() - s @ (csr(J) @ s)))
    monkeypatch.setattr(se.MaxCutEnv, "observation", lambda self: self.state.copy())
    return se


# ------------------------------------------------------------------------------------------------ graphs
def sym(n, r, c, w):
    A = np.zeros((n, n), dtype=np.int8)
    A[r, c] = w
    A[c, r] = w
    np.fill_diagonal(A, 0)
    return A


def random_edges(n, m, rng, weights=(-1, 1)):
    r = rng.integers(0, n, size=3 * m)
    c = rng.integers(0, n, size=3 * m)
    keep = r < c
    pairs = np.unique(np.stack([r[keep], c[keep]], 1), axis=0)
    pairs = pairs[rng.permutation(len(pairs))[:m]]
    return pairs[:, 0], pairs[:, 1], rng.choice(np.asarray(weights), size=len(pairs))


def ba_graph(n, m, seed):
    import networkx as nx
    g = nx.barabasi_albert_graph(n, m, seed=seed)
    e = np.array(g.edges())
    return sym(n, e[:, 0], e[:, 1], 1)


def torus(l1, l2, rng):
    """2-D toroidal grid with +-1 couplings (the shape of GSet G62 / G67 / G72 / G81)."""
    idx = np.arange(l1 * l2).reshape(l1, l2)
    r = np.concatenate([idx.ravel(), idx.ravel()])
    c = np.concatenate([np.roll(idx, 1, 0).ravel(), np.roll(idx, 1, 1).ravel()])
    return r, c, rng.choice(np.array([-1, 1]), size=len(r))


def dense_case(kind, n, G, seed):
    rng = np.random.default_rng(seed)
    if kind == "er":
        return np.stack([sym(n, *random_edges(n, int(0.15 * n * (n - 1) / 2), rng)) for _ in range(G)])
    if kind == "ba":
        return np.stack([ba_graph(n, 4, seed + g) for g in range(G)])
    if kind == "int":                                   # small integer weights
        return np.stack([sym(n, *random_edges(n, int(0.1 * n * (n - 1) / 2), rng, weights=(-3, -2, -1, 1, 2, 3)))
                         for _ in range(G)])
    if kind == "c4":                                    # 2000 vertices, 19 990 edges, +-1
        return np.stack([sym(n, *random_edges(n, 19990, rng)) for _ in range(G)])
    raise ValueError(kind)


def walk_actions(t, B, n, rng, prev):
    """random flips, with every third episode undoing its previous flip on odd steps (revisits)"""
    a = rng.integers(0, n, size=B).astype(np.int32)
    if t % 2 == 1:
        a[::3] = prev[::3]
    return a


def q_ok(q, ref):
    atol = Q_ATOL_FRAC * np.abs(ref).max(axis=-1, keepdims=True)
    return np.abs(q - ref) <= Q_RTOL * np.abs(ref) + atol


def state_arrays(env):
    return [env.spins, env.hfield, env.last_flip, env.diff_bits, env._ep, env.xn, env.xg]


# ------------------------------------------------------------------------------------------------ 1. dense parity
@pytest.mark.parametrize("kind,n", [("er", 20), ("ba", 200), ("int", 333), ("c4", 2000)])
def test_same_answers_as_dense_path(eng, wd, kind, n):
    from eco_dqn_b200 import _lib
    G, per = 2, 3
    Js = dense_case(kind, n, G, seed=n)
    gd = eng.GraphSet(Js)
    gsp = eng.SparseGraphSet(n, list(Js))
    assert torch.equal(gd.gscal, gsp.gscal) and torch.equal(gd.deg, gsp.deg)
    assert torch.equal(gd.gstat[:, :3], gsp.gstat[:, :3])
    dmax_d = eng._view(gd._ws, gd.c.dmax, 1, torch.float32, (1,))
    assert torch.equal(dmax_d, gsp.dmax)
    assert gsp.pm1_only == gd.pm1_only

    B, T = G * per, 2 * n
    steps = min(T, 60)
    gidx = np.repeat(np.arange(G, dtype=np.int32), per)
    rng = np.random.default_rng(7 + n)
    spins = (2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)
    ed, es = eng.BatchedSpinSystem(gd, B, T, 1.0 / n), eng.BatchedSpinSystem(gsp, B, T, 1.0 / n)
    for e in (ed, es):
        e.reset(spins=spins, graph_idx=gidx)
    for x, y in zip(state_arrays(ed), state_arrays(es)):
        assert torch.equal(x, y)
    prev = np.zeros(B, dtype=np.int32)
    for t in range(steps):
        acts = walk_actions(t, B, n, rng, prev)
        prev = acts
        a = torch.from_numpy(acts).cuda()
        rd, dd = (x.clone() for x in ed.step(a))
        rs, ds = es.step(a)
        assert torch.equal(rd.view(torch.int64), rs.view(torch.int64)) and torch.equal(dd, ds), (kind, n, t)
        for k, (x, y) in enumerate(zip(state_arrays(ed), state_arrays(es))):
            assert torch.equal(x, y), (kind, n, t, k)

    # the Q-network against the dense CUDA-core kernel, three norm_max modes; the fused argmax against the written Q
    for nm in (-1.0, None, 3.5):
        qd, _ = ed.q_values(eng.MPNNWeights(wd), norm_max=nm, impl=_lib.MPNN_SIMT)
        qs, acts = es.q_values(eng.MPNNWeights(wd), norm_max=nm)
        qd, qs = qd.cpu().numpy(), qs.cpu().numpy()
        assert q_ok(qs, qd).all(), (kind, n, nm, float(np.abs(qs - qd).max()))
        assert np.array_equal(acts.cpu().numpy(), qs.argmax(1))

    # Greedy rollouts
    for e in (ed, es):
        e.reset(spins=spins, graph_idx=gidx)
        e.rollout(policy="greedy")
    for x, y in zip(state_arrays(ed), state_arrays(es)):
        assert torch.equal(x, y)
    for x, y in zip(ed.results(), es.results()):
        assert torch.equal(x, y)


# ------------------------------------------------------------------------------------------------ 2. oracle, N > 2048
def big_case(n, seed):
    rng = np.random.default_rng(seed)
    if n == 10000:
        r, c, w = torus(100, 100, rng)
    elif n == 5000:                                     # G55 shape: 12 498 edges
        r, c, w = random_edges(n, 12498, rng)
    else:
        r, c, w = random_edges(n, 4 * n, rng)
    J = np.zeros((n, n))
    J[r, c] = w
    J[c, r] = w
    return (r, c, w), J


@pytest.mark.parametrize("n", [2500, 5000, 10000])
def test_beyond_dense_vs_oracle(eng, wd, sparse_oracle, n):
    from oracle.mpnn import mpnn_forward_blocked
    from oracle.rollout import greedy_baseline
    edges, J = big_case(n, seed=n)
    gs = eng.SparseGraphSet(n, [edges])
    B, T, steps = 2, 2 * n, 200
    br = 1.0 / n
    rng = np.random.default_rng(n + 1)
    spins = (2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)
    w = eng.MPNNWeights(wd)

    def compare(env, ors, r, d, t):
        ep = env.episodes()
        obs = env.observation().cpu().numpy()
        for b in range(B):
            o = ors[b]
            assert r is None or r[b].view(np.uint64) == np.float64(o.last_rew).view(np.uint64), (n, b, t)
            assert ep["score"][b] == o.score and ep["best_score"][b] == o.best_score, (n, b, t)
            assert d is None or bool(d[b]) == o.last_done
            assert np.array_equal(obs[b], o.state[:7].astype(np.float32)), (n, b, t)

    def oracle_envs():
        ors = [sparse_oracle.MaxCutEnv(J, T, br) for _ in range(B)]
        for o, s in zip(ors, spins):
            o.reset(s.astype(np.float64))
        return ors

    def ostep(o, a):
        _, o.last_rew, o.last_done, _ = o.step(int(a))

    def q_check(env, ors, acts=None):
        if n > 5000:
            return
        q, qa = env.q_values(w)
        q, qa = q.cpu().numpy(), qa.cpu().numpy()
        for b in range(B):
            ref = mpnn_forward_blocked(wd, ors[b].state[:7].T.astype(np.float32), J.astype(np.float32)).numpy()
            assert q_ok(q[b], ref).all(), (n, b, float(np.abs(q[b] - ref).max()))
            if acts is not None:
                assert ref.max() - ref[acts[b]] <= Q_RTOL * abs(ref.max()) + Q_ATOL_FRAC * np.abs(ref).max(), (n, b)

    # teacher-forced
    env = eng.BatchedSpinSystem(gs, B, T, br)
    env.reset(spins=spins)
    ors = oracle_envs()
    compare(env, ors, None, None, 0)
    q_check(env, ors)
    prev = np.zeros(B, dtype=np.int32)
    for t in range(steps):
        acts = walk_actions(t, B, n, rng, prev)
        prev = acts
        r, d = env.step(torch.from_numpy(acts).cuda())
        r, d = r.cpu().numpy(), d.cpu().numpy()
        for o, a in zip(ors, acts):
            ostep(o, a)
        compare(env, ors, r, d, t + 1)
    q_check(env, ors)

    # free-running network rollout, replayed through the oracle; every 20th action is an argmax of the oracle's Q
    env.reset(spins=spins)
    ha, hr, hs = env.rollout(w, n_steps=steps, record_history=True)
    ha, hr = ha.cpu().numpy(), hr.cpu().numpy()
    ors = oracle_envs()
    env2 = eng.BatchedSpinSystem(gs, B, T, br)
    env2.reset(spins=spins)
    for t in range(steps):
        if t % 20 == 0:
            q_check(env2, ors, ha[:, t])
        env2.step(torch.from_numpy(ha[:, t].copy()).cuda())
        for b in range(B):
            ostep(ors[b], ha[b, t])
            assert hr[b, t].view(np.uint64) == np.float64(ors[b].last_rew).view(np.uint64), (n, b, t)
    compare(env, ors, None, None, steps)
    bc, bs, st = env.results()
    assert np.array_equal(bc.cpu().numpy(), [o.best_solution for o in ors])
    assert np.array_equal(bs.cpu().numpy(), np.stack([o.best_spins for o in ors]).astype(np.int8))
    assert (st.cpu().numpy() == steps).all()

    # the Greedy baseline run to its stop
    env.reset(spins=spins)
    env.rollout(policy="greedy")
    cuts, gspins, gsteps = greedy_baseline(J, spins, T, br)
    bc, bs, st = env.results()
    assert np.array_equal(bc.cpu().numpy(), cuts)
    assert np.array_equal(bs.cpu().numpy(), gspins)
    assert np.array_equal(st.cpu().numpy(), gsteps)


# ------------------------------------------------------------------------------------------------ 3. invariants, G81 shape
def test_invariants_g81_shape(eng, wd):
    n, B, steps = 20000, 8, 500
    rng = np.random.default_rng(81)
    r, c, w = torus(100, 200, rng)
    gs = eng.SparseGraphSet(n, [(r, c, w)])
    A = sps.csr_matrix((np.concatenate([w, w]).astype(np.int64), (np.concatenate([r, c]), np.concatenate([c, r]))), shape=(n, n))
    env = eng.BatchedSpinSystem(gs, B, 2 * n, 1.0 / n)
    env.reset(spins=(2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8))
    env.rollout(eng.MPNNWeights(wd), n_steps=steps)
    s = env.spins[:, :n].cpu().numpy().astype(np.int64)
    h = env.hfield[:, :n].cpu().numpy().astype(np.int64)
    ep = env.episodes()
    obs = env.observation().cpu().numpy()
    bc, bs, st = (x.cpu().numpy() for x in env.results())
    mlr = float(gs.mlr[0])
    sumJ = int(A.sum())
    cut = lambda x: (sumJ - x @ (A @ x)) // 4
    for b in range(B):
        assert np.array_equal(h[b], A @ s[b])
        assert ep["cut"][b] == cut(s[b])
        assert bc[b] == ep["best_cut"][b] == cut(bs[b].astype(np.int64))
        dist = int((bs[b] != s[b]).sum())
        assert ep["dist"][b] == dist and obs[b, 4, 0] == dist
        assert np.array_equal(obs[b, 0], s[b].astype(np.float32))
        assert np.array_equal(obs[b, 1], ((s[b] * h[b]) / mlr).astype(np.float32))
        assert ep["n_improving"][b] == int((s[b] * h[b] > 0).sum())
        assert obs[b, 5, 0] == np.float32(ep["n_improving"][b] / n)
        assert st[b] == steps


# ------------------------------------------------------------------------------------------------ 4. drop-in
def env_args(n):
    from eco_dqn_b200.envs.utils import (DEFAULT_OBSERVABLES, RewardSignal, ExtraAction, OptimisationTarget, SpinBasis,
                                         Stopping)
    return {'observables': DEFAULT_OBSERVABLES, 'reward_signal': RewardSignal.BLS, 'extra_action': ExtraAction.NONE,
            'optimisation_target': OptimisationTarget.CUT, 'spin_basis': SpinBasis.SIGNED, 'norm_rewards': True,
            'memory_length': None, 'horizon_length': None, 'stag_punishment': None,
            'basin_reward': 1.0 / n, 'reversible_spins': True, 'stopping': Stopping.NORMAL}


def test_dropin_test_network_3000(eng, wd, sparse_oracle):
    from eco_dqn_b200.experiments.utils import test_network
    from oracle.rollout import greedy_baseline
    n, n_attempts, step_factor = 3000, 4, 0.1
    rng = np.random.default_rng(3000)
    graphs = [sym(n, *random_edges(n, 3 * n, rng)).astype(np.float64) for _ in range(2)]
    np.random.seed(11)
    res, raw = test_network(wd, env_args(n), graphs, "cuda", step_factor, n_attempts=n_attempts, return_raw=True)
    T = int(n * step_factor)
    for j in range(2):
        assert res["cut"][j] == max(raw["cuts"][j])
        init = np.stack(raw["init spins"][j])
        cuts, _, _ = greedy_baseline(graphs[j], init, T, 1.0 / n)
        assert np.array_equal(np.array(raw["greedy cuts"][j]), cuts)
        assert res["greedy (rand init) cut"][j] == cuts.max()
        c1, s1, _ = greedy_baseline(graphs[j], -np.ones((1, n)), T, 1.0 / n)
        assert res["greedy (+1 init) cut"][j] == c1[0]
        assert np.array_equal(res["greedy (+1 init) sol"][j], s1[0])


def test_dropin_load_mc_instances(eng, tmp_path):
    from eco_dqn_b200.experiments.utils import load_mc_instances_device
    n = 2500
    r, c, w = random_edges(n, 6000, np.random.default_rng(25))
    os.makedirs(tmp_path / "instances")
    with open(tmp_path / "instances" / "g.mc", "w") as f:
        f.write("%d %d\n" % (n, len(r)))
        for i, j, x in zip(r, c, w):
            f.write("%d %d %d\n" % (i + 1, j + 1, x))
    got = load_mc_instances_device(str(tmp_path), ["g"])
    want = eng.SparseGraphSet(n, [(r, c, w)])
    assert isinstance(got, eng.SparseGraphSet)
    for k in ("row_ptr", "col", "val", "gscal", "deg", "gstat"):
        assert torch.equal(getattr(got, k), getattr(want, k)), k


# ------------------------------------------------------------------------------------------------ 5. errors
def test_errors(eng, wd):
    from eco_dqn_b200.experiments.utils import test_network
    e1 = (np.array([0]), np.array([1]), np.array([1]))
    with pytest.raises(ValueError):
        eng.SparseGraphSet(32769, [e1])
    with pytest.raises(ValueError):                     # asymmetric (a scipy matrix is taken as stored)
        eng.SparseGraphSet(3000, [sps.csr_matrix(([1], ([0], [1])), shape=(3000, 3000))])
    with pytest.raises(ValueError):                     # non-zero diagonal
        eng.SparseGraphSet(3000, [(np.array([0, 5]), np.array([1, 5]), np.array([1, 1]))])
    with pytest.raises(ValueError):                     # no non-zero weighted degree
        eng.SparseGraphSet(3000, [(np.array([], dtype=int), np.array([], dtype=int), np.array([], dtype=int))])
    r, c, w = random_edges(3000, 9000, np.random.default_rng(1))
    with pytest.raises(NotImplementedError):            # real-valued couplings beyond 2048 vertices
        eng.SparseGraphSet(3000, [(r, c, w * 0.5)])
    with pytest.raises(NotImplementedError):
        test_network(wd, env_args(3000), [sym(3000, r, c, 1).astype(np.float64) * 0.5], "cuda", 0.01, n_attempts=1)
    with pytest.raises(NotImplementedError):            # MIN_CUT
        eng.SparseGraphSet(3000, [(r, c, w)], min_cut=True)
    gs = eng.SparseGraphSet(3000, [(r, c, w)])
    with pytest.raises(NotImplementedError):            # S2V-DQN
        eng.BatchedSpinSystem(gs, 2, 100, None, reversible_spins=False, dense_reward=True)
    with pytest.raises(NotImplementedError):
        eng.HostSession(1, 3000, 2, 100, None, wd)


def test_dropin_load_graph_set_networkx_pickle(eng, tmp_path):
    """A pickle of networkx graphs above 2048 vertices becomes a SparseGraphSet equal to one built from the same edges."""
    import pickle
    import networkx as nx
    from eco_dqn_b200.experiments.utils import load_graph_set_device
    n = 2500
    r, c, w = random_edges(n, 6000, np.random.default_rng(26))
    g = nx.Graph()
    g.add_nodes_from(range(n))
    g.add_weighted_edges_from(zip(r.tolist(), c.tolist(), w.tolist()))
    with open(tmp_path / "set.pkl", "wb") as f:
        pickle.dump([g, g], f)
    got = load_graph_set_device(str(tmp_path / "set.pkl"))
    want = eng.SparseGraphSet(n, [(r, c, w), (r, c, w)])
    assert isinstance(got, eng.SparseGraphSet)
    for k in ("row_ptr", "col", "val", "gscal", "deg", "gstat"):
        assert torch.equal(getattr(got, k), getattr(want, k)), k
