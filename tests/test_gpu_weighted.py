"""GPU tests of real-valued couplings (EdgeType.RANDOM): WeightedGraphSet, the fp64 environment, the MPNN on fp32(J), the
rollout, the Greedy baseline and the drop-in routing, against the golden vectors and the CPU oracle."""
import os
import random

import numpy as np
import pytest
import torch

from conftest import GOLDEN, golden_cases

pytestmark = pytest.mark.gpu

Q_RTOL = 1e-3
Q_ATOL_FRAC = 1e-4
ABS = 1e-9          # scores, normalised scores, rewards, cuts
OBS_RTOL = 2e-6     # observation rows (fp32 casts of fp64 values that may differ in the last bits)


def load(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def basin(z):
    b = float(z["basin_reward"])
    return None if b < 0 else b


@pytest.fixture(scope="module")
def eng():
    import eco_dqn_b200.engine as engine
    assert torch.cuda.is_available()
    return engine


@pytest.fixture(scope="module")
def wd():
    from oracle.mpnn import weights_from_npz
    return weights_from_npz(load("er20_g0"))


def random_graphs(n, G, seed, kind="er"):
    from eco_dqn_b200.envs.utils import EdgeType, RandomBarabasiAlbertGraphGenerator, RandomErdosRenyiGraphGenerator
    random.seed(seed)
    np.random.seed(seed)
    gen = (RandomErdosRenyiGraphGenerator(n, 0.15, EdgeType.RANDOM) if kind == "er"
           else RandomBarabasiAlbertGraphGenerator(n, 4, EdgeType.RANDOM))
    return np.stack([gen.get() for _ in range(G)])


def q_ok(q, ref):
    atol = Q_ATOL_FRAC * np.abs(ref).max(axis=-1, keepdims=True)
    return np.abs(q - ref) <= Q_RTOL * np.abs(ref) + atol


# ------------------------------------------------------------------------------------------------ integer graphs
@pytest.mark.parametrize("name", golden_cases())
def test_integer_graphs_through_weighted_path_bit_exact(eng, name):
    """Integer couplings as fp64: every sum is exact, so the weighted path must reproduce the reference bit for bit."""
    from oracle.mpnn import weights_from_npz
    z = load(name)
    T, n = int(z["T"]), int(z["n"])
    gs = eng.WeightedGraphSet(z["J"].astype(np.float64)[None])
    assert (float(gs.mlr[0]), float(gs.qn[0]), float(gs.lb[0])) == (float(z["mlr"]), float(z["qn"]), float(z["lb"]))
    B = z["init_spins"].shape[0]
    env = eng.BatchedSpinSystem(gs, B, T, basin(z))
    env.reset(spins=z["init_spins"], graph_idx=np.zeros(B, dtype=np.int32))
    w = eng.MPNNWeights(weights_from_npz(z))
    ep = env.episodes()
    assert np.array_equal(ep["score"], z["init_score"]) and np.array_equal(ep["cut"], z["init_cut"])
    k = z["obs"].shape[0]
    obs_steps = list(z["obs_steps"])
    rewards, dones = np.zeros((B, T)), np.zeros((B, T), dtype=np.uint8)
    scores, best_scores = np.zeros((B, T + 1)), np.zeros((B, T + 1))
    scores[:, 0], best_scores[:, 0] = ep["score"], ep["best_score"]
    acts = torch.from_numpy(z["actions"]).cuda()
    for t in range(T + 1):
        if t in obs_steps:
            i = obs_steps.index(t)
            assert np.array_equal(env.observation()[:k].cpu().numpy(), z["obs"][:, i]), (name, "obs at step", t)
            q, a = env.q_values(w)
            q, ref = q[:k].cpu().numpy(), z["q"][:, i]
            assert q_ok(q, ref).all(), (name, t, float(np.abs(q - ref).max()))
            assert np.array_equal(a[:k].cpu().numpy(), q.argmax(1))
        if t == T:
            break
        r, d = env.step(acts[:, t])
        rewards[:, t], dones[:, t] = r.cpu().numpy(), d.cpu().numpy()
        ep = env.episodes()
        scores[:, t + 1], best_scores[:, t + 1] = ep["score"], ep["best_score"]
    assert np.array_equal(rewards.view(np.uint64), z["rewards"].view(np.uint64)), "fp64 rewards must be bit-exact"
    assert np.array_equal(scores, z["scores"]) and np.array_equal(best_scores, z["best_scores"])
    assert np.array_equal(dones, z["dones"])
    bc, bs, st = env.results()
    assert bc.dtype == torch.float64
    assert np.array_equal(bc.cpu().numpy(), z["best_cut"])
    assert np.array_equal(bs.cpu().numpy(), z["best_spins"])
    assert np.array_equal(env.spins[:, :n].cpu().numpy(), z["final_spins"])
    assert (st.cpu().numpy() == T).all()


# ------------------------------------------------------------------------------------------------ real weights
def near_tie(env, best_before):
    """The oracle's score after a step within 1e-9 qn of its best score before the step: ulp noise decides the strict `>`
    of the BLS reward and the best tracking there, in the reference as well."""
    return abs(env.score - best_before) < 1e-9 * env.qn


@pytest.mark.parametrize("n,kind", [(20, "er"), (40, "ba"), (200, "er"), (333, "er"), (500, "ba")])
def test_real_weights_teacher_forced_vs_oracle(eng, n, kind):
    """Random, greedy and revisiting actions, several graphs per batch; each episode compared up to its first near tie.
    Revisiting episodes walk downhill and undo every other flip, so they return to visited configurations (basin-reward
    bookkeeping) without returning to the best one (which is a near tie by construction)."""
    from oracle.spin_env import MaxCutEnv
    G, per, T = 3, 6, 40
    Js = random_graphs(n, G, seed=1000 + n, kind=kind)
    gs = eng.WeightedGraphSet(Js)
    B = G * per
    gidx = np.repeat(np.arange(G, dtype=np.int32), per)
    rng = np.random.default_rng(n)
    spins = (2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)
    br = 1.0 / n
    env = eng.BatchedSpinSystem(gs, B, T, br)
    env.reset(spins=spins, graph_idx=gidx)
    ors = [MaxCutEnv(Js[gidx[b]], T, br) for b in range(B)]
    for b in range(B):
        ors[b].reset(spins[b].astype(np.float64))
    sc = gs.gscal.cpu().numpy()
    for g in range(G):
        o = ors[g * per]
        for got, want in zip(sc[g, :3], (o.mlr, o.qn, o.lb)):
            assert abs(got - want) <= 1e-12 * abs(want), (g, got, want)
    live = np.ones(B, dtype=bool)
    prev = np.zeros(B, dtype=np.int32)
    for t in range(T):
        acts = np.zeros(B, dtype=np.int32)
        for b in range(B):
            gains = ors[b]._gains(ors[b].spins)
            if b % 3 == 0:                                      # random
                acts[b] = rng.integers(0, n)
            elif b % 3 == 1:                                    # greedy while it improves, then random
                acts[b] = int(gains.argmax()) if gains.max() > 0 else rng.integers(0, n)
            else:                                               # revisiting: downhill flip, undo, downhill flip, ...
                acts[b] = prev[b] if t % 2 == 1 and t > 2 else int(gains.argmin())
        prev[:] = acts
        r, _ = env.step(torch.from_numpy(acts).cuda())
        r = r.cpu().numpy()
        ep = env.episodes()
        obs = env.observation().cpu().numpy()
        for b in range(B):
            if not live[b]:
                continue
            o = ors[b]
            best_before = o.best_obs_score
            _, rew, _, _ = o.step(int(acts[b]))
            if near_tie(o, best_before):
                live[b] = False
                continue
            assert abs(r[b] - rew) <= ABS, (n, b, t, r[b], rew)
            assert abs(ep["score"][b] - o.score) <= ABS and abs(ep["nscore"][b] - o.nscore) <= ABS, (n, b, t)
            assert abs(ep["best_score"][b] - o.best_score) <= ABS
            want = o.state.astype(np.float32)
            assert np.allclose(obs[b], want, rtol=OBS_RTOL, atol=OBS_RTOL), (n, b, t, np.abs(obs[b] - want).max())
    bc, bs, _ = env.results()
    bc, bs = bc.cpu().numpy(), bs.cpu().numpy()
    for b in np.nonzero(live)[0]:
        assert abs(bc[b] - ors[b].best_solution) <= ABS
        assert np.array_equal(bs[b], ors[b].best_spins.astype(np.int8))
    print("n=%d: %d of %d episodes stopped at a near tie" % (n, int((~live).sum()), B))
    assert (~live).sum() < B / 2


@pytest.mark.parametrize("n", [40, 200, 333])
def test_real_weights_free_running_rollout_vs_oracle(eng, wd, n):
    """The device's own actions replayed through the oracle: rewards / scores agree and every action maximises the
    oracle's Q within the Q contract (each episode up to its first near tie)."""
    from oracle.rollout import rollout as cpu_rollout
    G, per, T = 2, 3, min(2 * n, 60)
    Js = random_graphs(n, G, seed=2000 + n)
    gs = eng.WeightedGraphSet(Js)
    B = G * per
    gidx = np.repeat(np.arange(G, dtype=np.int32), per)
    spins = (2 * np.random.default_rng(n).integers(0, 2, size=(B, n)) - 1).astype(np.int8)
    br = 1.0 / n
    env = eng.BatchedSpinSystem(gs, B, T, br)
    env.reset(spins=spins, graph_idx=gidx)
    ha, hr, hs = env.rollout(eng.MPNNWeights(wd), record_history=True)
    ha, hr, hs = ha.cpu().numpy(), hr.cpu().numpy(), hs.cpu().numpy()
    stopped = 0
    for g in range(G):
        sl = slice(g * per, (g + 1) * per)
        ok_q = []

        def hook(t, qs):
            qs = qs.numpy()
            picked = qs[np.arange(qs.shape[0]), ha[sl][:, t]]
            qmax = qs.max(1)
            ok_q.append(qmax - picked <= Q_RTOL * np.abs(qmax) + Q_ATOL_FRAC * np.abs(qs).max(1))

        ref = cpu_rollout(Js[g], wd, spins[sl], T, br, forced_actions=ha[sl], q_hook=hook)
        # first near tie of each episode: score within 1e-9 qn of the best score before the step
        qn = max(1, np.sum(Js[g] * (Js[g] > 0)) / 2)
        best_before = np.maximum.accumulate(ref["scores"], axis=1)[:, :-1]
        tie = np.abs(ref["scores"][:, 1:] - best_before) < 1e-9 * qn
        for e in range(per):
            stop = int(np.argmax(tie[e])) if tie[e].any() else T
            stopped += stop < T
            assert np.abs(hr[sl][e, :stop] - ref["rewards"][e, :stop]).max(initial=0) <= ABS
            assert np.abs(hs[sl][e, :stop] - ref["scores"][e, 1:stop + 1]).max(initial=0) <= ABS
            assert all(ok_q[t][e] for t in range(stop)), (n, g, e)
    print("n=%d: %d of %d episodes stopped at a near tie" % (n, stopped, B))
    assert stopped < B / 2


@pytest.mark.parametrize("n", [20, 200, 500])
def test_real_weights_greedy_vs_oracle(eng, n):
    from oracle.rollout import greedy_baseline
    G, per, T = 2, 4, 2 * n
    Js = random_graphs(n, G, seed=3000 + n)
    gs = eng.WeightedGraphSet(Js)
    for start in ("random", "minus_one"):
        B = G * per
        gidx = np.repeat(np.arange(G, dtype=np.int32), per)
        if start == "random":
            spins = (2 * np.random.default_rng(n).integers(0, 2, size=(B, n)) - 1).astype(np.int8)
        else:
            spins = -np.ones((B, n), dtype=np.int8)
        env = eng.BatchedSpinSystem(gs, B, T, None)
        env.reset(spins=spins, graph_idx=gidx)
        env.rollout(policy="greedy")
        bc, bs, st = (x.cpu().numpy() for x in env.results())
        for g in range(G):
            sl = slice(g * per, (g + 1) * per)
            cuts, sp, steps = greedy_baseline(Js[g], spins[sl].astype(np.float64), T)
            assert np.array_equal(st[sl], steps), (n, start, g)
            assert np.array_equal(bs[sl], sp), (n, start, g)
            assert np.abs(bc[sl] - cuts).max() <= ABS


# ------------------------------------------------------------------------------------------------ drop-in surface
def env_args(**kw):
    from eco_dqn_b200.envs.utils import (DEFAULT_OBSERVABLES, RewardSignal, ExtraAction, OptimisationTarget, SpinBasis,
                                         Stopping)
    a = {'observables': DEFAULT_OBSERVABLES, 'reward_signal': RewardSignal.BLS, 'extra_action': ExtraAction.NONE,
         'optimisation_target': OptimisationTarget.CUT, 'spin_basis': SpinBasis.SIGNED, 'norm_rewards': True,
         'memory_length': None, 'horizon_length': None, 'stag_punishment': None, 'basin_reward': 1 / 20,
         'reversible_spins': True, 'stopping': Stopping.NORMAL}
    a.update(kw)
    return a


def test_dropin_test_network_real_graphs(wd):
    from eco_dqn_b200.envs.utils import calculate_cut
    from eco_dqn_b200.experiments.utils import test_network
    from oracle.spin_env import MaxCutEnv
    graphs = list(random_graphs(20, 4, seed=77))
    n_att = 5
    np.random.seed(11)
    res, raw = test_network(dict(wd), env_args(), graphs, "cuda", 2, n_attempts=n_att, return_raw=True)
    assert list(res.columns) == ["cut", "sol", "mean cut", "greedy (+1 init) cut", "greedy (+1 init) sol",
                                 "greedy (rand init) cut", "greedy (rand init) sol", "greedy (rand init) mean cut", "time"]
    for j, J in enumerate(graphs):
        assert abs(res["cut"][j] - calculate_cut(res["sol"][j], J)) <= ABS
        # greedy columns: the oracle's Greedy from the same global-RNG starts
        starts = np.array(raw["init spins"][j])
        g_cuts = []
        for s in starts:
            o = MaxCutEnv(J, 40, None)
            o.reset(s)
            o.greedy_solve()
            g_cuts.append(o.best_solution)
        assert np.abs(np.array(raw["greedy cuts"][j]) - np.array(g_cuts)).max() <= ABS
        o = MaxCutEnv(J, 40, None)
        o.reset(-np.ones(20))
        o.greedy_solve()
        assert abs(res["greedy (+1 init) cut"][j] - o.best_solution) <= ABS
        assert np.array_equal(res["greedy (+1 init) sol"][j], o.best_spins)
    np.random.seed(11)
    for j in range(len(graphs)):        # the starts are the reference's draws: N for the constructor, N per attempt
        np.random.randint(2, size=20)
        want = np.stack([2 * np.random.randint(2, size=20) - 1 for _ in range(n_att)])
        assert np.array_equal(np.array(raw["init spins"][j]), want)


def test_dropin_make_single_graph_steps_match_oracle():
    from eco_dqn_b200.envs.core import make
    from eco_dqn_b200.envs.utils import SingleGraphGenerator, RewardSignal, ExtraAction, OptimisationTarget
    from oracle.spin_env import MaxCutEnv
    J = random_graphs(20, 1, seed=5)[0]
    env = make("SpinSystem", SingleGraphGenerator(J), 30, reward_signal=RewardSignal.BLS, extra_action=ExtraAction.NONE,
               optimisation_target=OptimisationTarget.CUT, norm_rewards=True, basin_reward=1 / 20)
    s0 = 2 * np.random.default_rng(3).integers(0, 2, size=20) - 1
    env.reset(spins=s0)
    o = MaxCutEnv(J, 30, 1 / 20)
    o.reset(s0.astype(np.float64))
    rng = np.random.default_rng(4)
    for t in range(30):
        a = int(rng.integers(0, 20))
        ob, r, done, _ = env.step(a)
        best_before = o.best_obs_score
        ob_o, r_o, done_o, _ = o.step(a)
        if near_tie(o, best_before):
            break
        assert abs(r - r_o) <= ABS and done == done_o
        assert abs(env.score - o.score) <= ABS
        assert np.allclose(ob[:7], ob_o[:7].astype(np.float32), rtol=OBS_RTOL, atol=OBS_RTOL)
        assert np.array_equal(ob[7:], J)
    assert abs(env.best_solution - o.best_solution) <= ABS


def test_dropin_unsupported_weighted_configurations(wd):
    from eco_dqn_b200.envs.core import make
    from eco_dqn_b200.envs.utils import (SingleGraphGenerator, RewardSignal, ExtraAction, OptimisationTarget, Observable)
    import eco_dqn_b200.engine as engine
    J = random_graphs(20, 1, seed=6)[0]
    with pytest.raises(NotImplementedError):
        make("SpinSystem", SingleGraphGenerator(J), 20, reward_signal=RewardSignal.BLS, extra_action=ExtraAction.NONE,
             optimisation_target=OptimisationTarget.MIN_CUT, norm_rewards=True)
    with pytest.raises(NotImplementedError):          # S2V-DQN: irreversible spins, dense reward
        make("SpinSystem", SingleGraphGenerator(J), 20, observables=[Observable.SPIN_STATE],
             reward_signal=RewardSignal.DENSE, extra_action=ExtraAction.NONE, optimisation_target=OptimisationTarget.CUT,
             norm_rewards=True, reversible_spins=False)
    with pytest.raises(NotImplementedError):
        engine.GraphSet(J[None])
    with pytest.raises(NotImplementedError):
        engine.HostSession(1, 20, 2, 20, None, wd).rollout(J[None], np.zeros(2, dtype=np.int32),
                                                           -np.ones((2, 20), dtype=np.int8), np.zeros(2, dtype=np.int32))
    from eco_dqn_b200.agents.dqn.dqn import DQN
    from eco_dqn_b200.networks.mpnn import MPNN
    env = make("SpinSystem", SingleGraphGenerator(J), 20, reward_signal=RewardSignal.BLS, extra_action=ExtraAction.NONE,
               optimisation_target=OptimisationTarget.CUT, norm_rewards=True, basin_reward=1 / 20)
    with pytest.raises(NotImplementedError):
        DQN([env], lambda: MPNN(), replay_buffer_size=100, minibatch_size=4, logging=False, n_envs=2)


def test_weighted_graph_validation(eng):
    J = random_graphs(20, 1, seed=8)[0]
    bad = J.copy(); bad[0, 1] += 0.5
    with pytest.raises(ValueError):
        eng.WeightedGraphSet(bad[None])
    bad = J.copy(); bad[3, 3] = 0.25
    with pytest.raises(ValueError):
        eng.WeightedGraphSet(bad[None])
    bad = J.copy(); bad[0, 1] = bad[1, 0] = np.nan
    with pytest.raises(ValueError):
        eng.WeightedGraphSet(bad[None])
    with pytest.raises(ValueError):
        eng.WeightedGraphSet(np.zeros((1, 20, 20)))
    with pytest.raises(ValueError):
        eng.WeightedGraphSet(np.zeros((1, 2049, 2049)))
    from eco_dqn_b200 import _lib
    gs = eng.WeightedGraphSet(J[None])
    env = eng.BatchedSpinSystem(gs, 2, 10, None)
    env.reset()
    from oracle.mpnn import weights_from_npz
    w = eng.MPNNWeights(weights_from_npz(load("er20_g0")))
    with pytest.raises(NotImplementedError):          # the tensor-core MPNN is {-1,0,1}-only
        env.q_values(w, impl=_lib.MPNN_TCGEN05)


# ------------------------------------------------------------------------------------------------ full size
def test_full_size_invariants(eng, wd):
    """B = 4096 episodes on 64 ER-200 RANDOM graphs: h = J s in fp64, best cut = cut(best spins), the Hamming distance row,
    and the fused argmax against the written Q."""
    n, G, B, T = 200, 64, 4096, 30
    Js = random_graphs(n, G, seed=9)
    gs = eng.WeightedGraphSet(Js)
    gidx = (np.arange(B) % G).astype(np.int32)
    env = eng.BatchedSpinSystem(gs, B, T, 1.0 / n)
    np.random.seed(10)
    env.reset(graph_idx=gidx)
    w = eng.MPNNWeights(wd)
    env.rollout(w, n_steps=20)
    J = torch.from_numpy(Js).cuda()[torch.from_numpy(gidx).cuda().long()]          # [B, n, n] fp64
    s = env.spins[:, :n].double()
    h = torch.bmm(J, s[:, :, None])[:, :, 0]
    assert (h - env.hfield[:, :n]).abs().max().item() <= ABS
    bc, bs, _ = env.results()
    bsd = bs.double()
    cut = 0.25 * (J * (1 - bsd[:, :, None] * bsd[:, None, :])).sum((1, 2))
    assert (cut - bc).abs().max().item() <= ABS
    obs = env.observation()
    dist = (bs != env.spins[:, :n]).sum(1).float()
    assert torch.equal(obs[:, 4, 0], dist)
    q, a = env.q_values(w, norm_max=-1)
    assert torch.equal(a.long(), q.argmax(1))
