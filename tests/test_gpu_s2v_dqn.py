"""GPU tests of S2V-DQN training (irreversible spins, spin-only observation, dense reward, MPNN(n_obs_in=1)) on the device
trainer: the masked TD-target and exploration kernels against torch restatements, the 1-observable update against autograd
and torch.optim.Adam, the captured update / acting step, and learn() end to end."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import GOLDEN

pytestmark = pytest.mark.gpu


def s2v_env_args():
    from eco_dqn_b200.envs.utils import Observable, RewardSignal, ExtraAction, OptimisationTarget, SpinBasis
    return {'observables': [Observable.SPIN_STATE], 'reward_signal': RewardSignal.DENSE, 'extra_action': ExtraAction.NONE,
            'optimisation_target': OptimisationTarget.CUT, 'spin_basis': SpinBasis.SIGNED, 'norm_rewards': True,
            'memory_length': None, 'horizon_length': None, 'stag_punishment': None, 'basin_reward': None,
            'reversible_spins': False}


def make_s2v_agent(tmp_path, graphs, T, **kw):
    import eco_dqn_b200.envs.core as ising_env
    from eco_dqn_b200.envs.utils import SetGraphGenerator
    from eco_dqn_b200.networks.mpnn import MPNN
    from eco_dqn_b200.agents.dqn.dqn import DQN
    from eco_dqn_b200.agents.dqn.utils import TestMetric
    env = ising_env.make("SpinSystem", SetGraphGenerator([g.astype(np.float64) for g in graphs], ordered=True), T,
                         **s2v_env_args())
    args = dict(double_dqn=True, gamma=0.95, update_learning_rate=False, initial_learning_rate=1e-4, minibatch_size=16,
                replay_buffer_size=400, replay_start_size=64, logging=False, seed=3, test_metric=TestMetric.BEST,
                test_save_path=str(tmp_path / "scores"), network_save_path=str(tmp_path / "net"), n_envs=4)
    args.update(kw)
    return DQN([env], lambda: MPNN(n_obs_in=1), **args)


def er20(k=6):
    return list(np.load(os.path.join(GOLDEN, "graphsets.npz"))["er20"][:k])


def random_pm1_graphs(n, p, G, rng):
    Js = np.zeros((G, n, n), dtype=np.int8)
    for g in range(G):
        up = np.triu(rng.random((n, n)) < p, 1)
        a = (up * np.where(rng.random((n, n)) < 0.5, -1, 1)).astype(np.int8)
        Js[g] = a + a.T
    Js[:, 0, 1] = Js[:, 1, 0] = 1
    return Js


def padded_cols_zero(shadow):
    sd = shadow.state_dict()
    return bool((sd["node_init_embedding_layer.0.weight"][:, 1:] == 0).all()) and \
        bool((sd["edge_embedding_layer.edge_embedding_NN.weight"][:, 2:] == 0).all())


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [20, 40, 200, 333])
@pytest.mark.parametrize("double_dqn", [True, False])
@pytest.mark.parametrize("clip", [True, False])
def test_masked_td_target_matches_torch(n, double_dqn, clip):
    """eco_dqn_masked_td_target against masked_fill(-1000) -> argmax -> gather -> clamp -> r + (1 - d) gamma q on the same Q
    tensors: masks from one -1 spin left to all -1, all-+1 terminal rows, exact ties in Q; chosen index equal, td bit-identical."""
    from eco_dqn_b200._lib import lib, check
    import eco_dqn_b200.engine as eng
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(n + 2 * double_dqn + clip)
    NP = (n + 15) // 16 * 16
    B = 96
    q_on = torch.tensor(np.round(rng.standard_normal((B, NP)) * 3) / 2, dtype=torch.float32, device=dev)   # many exact ties
    q_tg = torch.tensor(np.round(rng.standard_normal((B, NP)) * 3) / 2, dtype=torch.float32, device=dev)
    q_tg[::7] = -abs(q_tg[::7]) - 0.5                                         # rows where every target is negative (clip)
    q_on[::11] = 1.0                                                          # a whole row tied
    spins = np.ones((B, n), dtype=np.float32)
    for b in range(B):
        k = [1, n, 0][b % 3] if b < 6 else int(rng.integers(1, n + 1))      # one left, all -1, none (terminal) ...
        spins[b, rng.permutation(n)[:k]] = -1.0
    xn_next = torch.zeros(B, 3, NP, device=dev)
    xn_next[:, 0, :n] = torch.tensor(spins, device=dev)
    xn_next[:, 1:, :n] = torch.randn(B, 2, n, device=dev)
    reward = torch.tensor(rng.standard_normal(B).astype(np.float32), device=dev)
    done = torch.tensor((spins == 1).all(1).astype(np.float32), device=dev)
    done[5::13] = 1.0
    gamma = 0.95
    td = torch.full((B,), float("nan"), device=dev)
    chosen = torch.full((B,), -1, dtype=torch.int32, device=dev)
    check(lib().eco_dqn_masked_td_target(B, n, NP, eng._ptr(q_on), eng._ptr(q_tg), eng._ptr(xn_next), eng._ptr(reward),
                                         eng._ptr(done), gamma, int(double_dqn), int(clip), eng._ptr(td), eng._ptr(chosen),
                                         eng._stream()))
    mask = xn_next[:, 0, :n] != -1
    if double_dqn:
        a = q_on[:, :n].masked_fill(mask, -1000.0).argmax(1, True)
        v = q_tg[:, :n].gather(1, a)
    else:
        masked = q_tg[:, :n].masked_fill(mask, -1000.0)
        a = masked.argmax(1, True)
        v = masked.max(1, True)[0]
    if clip:
        v = v.clamp(min=0)
    ref = reward.unsqueeze(1) + (1 - done.unsqueeze(1)) * gamma * v
    torch.cuda.synchronize()
    assert torch.equal(chosen.long(), a.reshape(-1))
    assert torch.equal(td.view(torch.int32), ref.reshape(-1).view(torch.int32))


# ---------------------------------------------------------------------------------------------------------------------
def _explore(env, q, u, eps, ready):
    from eco_dqn_b200._lib import lib, check
    import eco_dqn_b200.engine as eng
    act = torch.full((env.B,), -1, dtype=torch.int32, device=env.device)
    check(lib().eco_dqn_masked_explore(C.byref(env.c), eng._ptr(q), eng._ptr(u), eng._ptr(eps), eng._ptr(ready), eng._ptr(act),
                                       eng._stream()))
    return act


def test_masked_explore_kernel():
    """eco_dqn_masked_explore: every action is a spin still at -1; eps = 0 and ready gives the masked argmax; eps = 1 is
    uniform over the allowed set (chi-square over >= 20 000 draws per pattern, c = 1 included); c = 0 gives action 0; the same
    generator seed gives the same actions."""
    from scipy.stats import chisquare
    from eco_dqn_b200._lib import lib, check
    import eco_dqn_b200.engine as eng
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(11)
    n = 40
    gs = eng.GraphSet(random_pm1_graphs(n, 0.15, 1, rng), device=dev)
    patterns = []
    for c in (1, 7, 23, 40, 0):
        s = np.ones(n, dtype=np.int8)
        s[rng.permutation(n)[:c]] = -1
        patterns.append(s)
    reps = 1024
    B = reps * len(patterns)
    env = eng.BatchedSpinSystem(gs, B, n, None, reversible_spins=False, dense_reward=True)
    env.reset(spins=np.repeat(np.stack(patterns), reps, axis=0), graph_idx=np.zeros(B, dtype=np.int32))
    sp = env.spins[:, :n].cpu().numpy()
    q = torch.tensor(np.round(rng.standard_normal((B, env.NP)) * 2) / 2, dtype=torch.float32, device=dev)
    one, zero = torch.ones(1, device=dev), torch.zeros(1, device=dev)
    t_ready, f_ready = torch.ones(1, dtype=torch.bool, device=dev), torch.zeros(1, dtype=torch.bool, device=dev)
    gen = torch.Generator(device=dev).manual_seed(5)

    # greedy
    a = _explore(env, q, torch.rand(B, 2, device=dev, generator=gen), zero, t_ready)
    ref = torch.zeros(B, dtype=torch.int32, device=dev)
    check(lib().eco_env_masked_argmax(C.byref(env.c), eng._ptr(q), eng._ptr(ref), eng._stream()))
    assert torch.equal(a, ref)
    # eps = 0 but training not ready: explores
    a = _explore(env, q, torch.rand(B, 2, device=dev, generator=gen), zero, f_ready).cpu().numpy()
    assert not np.array_equal(a, ref.cpu().numpy())
    # eps = 1: uniform over the allowed set
    draws = 20
    counts = [np.zeros(n, dtype=np.int64) for _ in patterns]
    for _ in range(draws):
        a = _explore(env, q, torch.rand(B, 2, device=dev, generator=gen), one, t_ready).cpu().numpy()
        for pi in range(len(patterns)):
            ap = a[pi * reps:(pi + 1) * reps]
            if pi == len(patterns) - 1:
                assert (ap == 0).all()                                  # c = 0: action 0
                continue
            assert (sp[np.arange(pi * reps, (pi + 1) * reps), ap] == -1).all()
            counts[pi] += np.bincount(ap, minlength=n)
    for pi, s in enumerate(patterns[:-1]):
        allowed = np.flatnonzero(s == -1)
        assert counts[pi].sum() == draws * reps >= 20000 and counts[pi][s == 1].sum() == 0
        if len(allowed) > 1:
            assert chisquare(counts[pi][allowed]).pvalue > 1e-4, (pi, counts[pi][allowed])
    # reproducible from the generator seed
    outs = []
    for _ in range(2):
        g2 = torch.Generator(device=dev).manual_seed(123)
        outs.append(_explore(env, q, torch.rand(B, 2, device=dev, generator=g2), torch.full((1,), 0.5, device=dev), t_ready))
    assert torch.equal(outs[0], outs[1])


# ---------------------------------------------------------------------------------------------------------------------
def _flat_views(flat):
    import eco_dqn_b200.engine as eng
    out, off = {}, 0
    for key, shp in zip(eng.STATE_DICT_KEYS, eng.STATE_DICT_SHAPES):
        cnt = int(np.prod(shp))
        out[key] = flat[off:off + cnt].view(shp)
        off += cnt
    return out


@pytest.mark.parametrize("n,p,B,loss_name", [(17, 0.3, 5, "mse"), (40, 0.15, 16, "huber"), (200, 0.04, 9, "mse")])
def test_s2v_update_matches_autograd_and_torch_adam(n, p, B, loss_name):
    """eco_mpnn_grad_obs on the padded shadow of an MPNN(n_obs_in=1) against autograd through the module on [B, 1 + N, N]:
    loss 1e-5 rel, every gradient tensor 1e-4 of its largest entry, the padded columns' gradient exactly 0.0; Adam on the
    shadow within 2e-6 of torch.optim.Adam on the 1-observable module; after 50 updates with weight decay the padded columns
    are exactly 0.0."""
    from eco_dqn_b200 import _lib
    from eco_dqn_b200._lib import lib, check
    import eco_dqn_b200.engine as eng
    from eco_dqn_b200.networks.mpnn import MPNN
    from eco_dqn_b200.agents.dqn.dqn import padded_shadow
    from eco_dqn_b200.agents.dqn.utils import KernelAdam
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(3 * n + B)
    torch.manual_seed(n)
    G = 3
    Js = random_pm1_graphs(n, p, G, rng)
    gs = eng.GraphSet(Js, device=dev)
    NP = gs.NP
    net = MPNN(n_obs_in=1).to(dev)
    with torch.no_grad():
        for q in net.parameters():
            q.copy_(torch.randn_like(q) * (0.3 if q.dim() > 1 else 0.1))
    ref_net = MPNN(n_obs_in=1).to(dev)
    ref_net.load_state_dict(net.state_dict())
    shadow = padded_shadow(net, dev)
    gidx = torch.tensor(rng.integers(0, G, size=B), dtype=torch.int32, device=dev)
    xn = torch.zeros(B, 3, NP, device=dev)
    xn[:, 0, :n] = torch.tensor(np.where(rng.random((B, n)) < 0.5, -1.0, 1.0).astype(np.float32), device=dev)
    xn[:, 1:, :n] = torch.randn(B, 2, n, device=dev)                # rows the 1-observable network does not see
    xg = torch.randn(B, 4, device=dev)
    actions = torch.tensor(rng.integers(0, n, size=B), dtype=torch.int32, device=dev)
    targets = torch.tensor(rng.standard_normal(B).astype(np.float32) * 3, device=dev)
    norm_max = float(max(1, (Js != 0).sum(1)[gidx.cpu().numpy()].max()))
    loss_kind = {"mse": _lib.LOSS_MSE, "huber": _lib.LOSS_HUBER}[loss_name]

    adj = torch.tensor(Js.astype(np.float32), device=dev)[gidx.long()]
    obs = torch.cat([xn[:, :1, :n], adj], dim=1)
    qv = ref_net(obs).gather(1, actions.long().unsqueeze(1)).squeeze(1)
    loss_ref = {"mse": F.mse_loss, "huber": F.smooth_l1_loss}[loss_name](qv, targets, reduction="mean")
    ref_net.zero_grad()
    loss_ref.backward()

    w = shadow.engine_weights(dev)
    assert w.aliases
    scratch = torch.empty(lib().eco_mpnn_grad_scratch_bytes(B, n), dtype=torch.uint8, device=dev)

    def grad_call():
        flat = torch.full((_lib.MPNN_N_PARAMS,), float("nan"), device=dev)
        loss = torch.full((1,), float("nan"), device=dev)
        check(lib().eco_mpnn_grad_obs(C.byref(gs.c), C.byref(w.c), B, eng._ptr(gidx), eng._ptr(xn), eng._ptr(xg), norm_max,
                                      eng._ptr(actions), eng._ptr(targets), loss_kind, 1, eng._ptr(loss), eng._ptr(flat),
                                      eng._ptr(scratch), None, eng._stream()))
        return loss, flat

    loss, flat = grad_call()
    loss_r = float(loss_ref.detach())
    assert abs(float(loss) - loss_r) <= 1e-5 * abs(loss_r) + 1e-7
    views = _flat_views(flat)
    assert torch.equal(views["node_init_embedding_layer.0.weight"][:, 1:], torch.zeros(64, 6, device=dev))
    assert torch.equal(views["edge_embedding_layer.edge_embedding_NN.weight"][:, 2:], torch.zeros(63, 6, device=dev))
    for key, pr in ref_net.named_parameters():
        gk = views[key][..., :pr.shape[-1]] if pr.dim() > 1 else views[key]
        gr = pr.grad
        assert torch.isfinite(gk).all(), key
        assert float((gk - gr).abs().max()) <= 1e-4 * float(gr.abs().max()) + 1e-8, key

    # one Adam step on the shadow vs torch.optim.Adam on the 1-observable module, same gradient
    opt = KernelAdam(shadow, lr=3e-3, eps=1e-8, weight_decay=0.01)
    opt_ref = torch.optim.Adam(ref_net.parameters(), lr=3e-3, eps=1e-8, weight_decay=0.01)
    for key, sp in shadow.named_parameters():
        sp.grad = views[key]
    for key, pr in ref_net.named_parameters():
        pr.grad = (views[key][..., :pr.shape[-1]] if pr.dim() > 1 else views[key]).clone()
    opt.step()
    opt_ref.step()
    for (key, pa), pb in zip(net.named_parameters(), ref_net.parameters()):
        assert pa.shape == pb.shape
        assert torch.allclose(pa, pb, rtol=2e-6, atol=1e-8), (key, float((pa - pb).abs().max()))
    # 50 more updates with weight decay: the padded columns stay exactly 0.0
    for _ in range(50):
        loss, flat = grad_call()
        for key, sp in shadow.named_parameters():
            sp.grad = _flat_views(flat)[key]
        opt.step()
    torch.cuda.synchronize()
    assert padded_cols_zero(shadow) and opt.steps == 51
    assert torch.equal(net.state_dict()["node_init_embedding_layer.0.weight"],
                       shadow.state_dict()["node_init_embedding_layer.0.weight"][:, :1])


# ---------------------------------------------------------------------------------------------------------------------
def _fill_replay(agent, timesteps):
    start = agent.replay_start_size
    agent.replay_start_size = 10 ** 9
    agent.learn(timesteps=timesteps)
    agent.replay_start_size = start


def test_s2v_captured_update_equals_eager_update(tmp_path):
    """The captured S2V update (network forwards, masked TD-target kernel, eco_mpnn_grad_obs, Adam) gives bit for bit the
    parameters of the same updates launched eagerly, across a learning-rate change and a target sync."""
    agent = make_s2v_agent(tmp_path, er20(), 20, n_envs=8, init_weight_std=0.05, minibatch_size=16, replay_buffer_size=1000,
                           replay_start_size=64, weight_decay=0.01)
    _fill_replay(agent, 320)
    gen = torch.Generator(device="cuda").manual_seed(3)
    idxs = [agent.replay_buffer.sample_indices(16, gen) for _ in range(6)]
    o = agent.optimizer
    st0 = ([p.detach().clone() for p in agent._qnet.parameters()], o.exp_avg.clone(), o.exp_avg_sq.clone(), o.step_dev.clone())
    tgt0 = {k: v.clone() for k, v in agent._qnet_target.state_dict().items()}

    def run(step_fn):
        with torch.no_grad():
            for p, q in zip(agent._qnet.parameters(), st0[0]):
                p.copy_(q)
            o.exp_avg.copy_(st0[1]); o.exp_avg_sq.copy_(st0[2]); o.step_dev.copy_(st0[3])
        agent._qnet.engine_weights(agent.device).repack()
        agent._qnet_target.load_state_dict(tgt0)
        agent._qnet_target.engine_weights(agent.device)
        out = []
        for k, idx in enumerate(idxs):
            if k == 2:
                o.param_groups[0]['lr'] = 3e-4
            if k == 4:
                agent.target_network.load_state_dict(agent.network.state_dict())    # through the 1-observable modules
                agent._qnet_target.engine_weights(agent.device)
            out.append(float(step_fn(idx)))
        o.param_groups[0]['lr'] = 1e-4
        return out, [p.detach().clone() for p in agent._qnet.parameters()]

    l_eager, p_eager = run(lambda idx: agent._update(agent.replay_buffer.gather(idx)))
    assert agent._cg is None
    l_graph, p_graph = run(agent._train_step_device)
    assert agent._cg is not None and l_eager == l_graph
    for a, b in zip(p_eager, p_graph):
        assert torch.equal(a, b)
    assert not torch.equal(p_eager[2], st0[0][2]) and padded_cols_zero(agent._qnet)


def _check_episodes(agent, n_rows, n, E):
    rb = agent.replay_buffer
    xn, xn2 = rb.xn[:n_rows].cpu(), rb.xn_next[:n_rows].cpu()
    act, done, rew = rb.action[:n_rows].cpu(), rb.done[:n_rows].cpu(), rb.reward[:n_rows].cpu().double()
    graph = rb.graph[:n_rows].cpu()
    for e in range(E):
        rows = torch.arange(e, n_rows, E)
        for ep in range(len(rows) // n):
            r = rows[ep * n:(ep + 1) * n]
            assert (xn[r[0], 0, :n] == -1).all()                             # all -1 start
            for i in r.tolist():
                a = int(act[i])
                assert xn[i, 0, a] == -1                                     # an allowed action
                expect = xn[i, 0, :n].clone()
                expect[a] = 1.0
                assert torch.equal(xn2[i, 0, :n], expect)
            assert len(set(act[r].tolist())) == n                            # N distinct actions
            assert done[r[:-1]].sum() == 0 and done[r[-1]] == 1
            # dense reward: the normalised cut change of the flip (spinsystem.py:435-436)
            J = agent._graphs.J[int(graph[r[0]]), :n, :n].cpu().double()
            cut = lambda s: float(((1 - torch.outer(s, s)) * J).sum() / 4)
            s0 = xn[r, 0, :n].double()
            s1 = xn2[r, 0, :n].double()
            deg = float(agent._graphs.gscal[int(graph[r[0]]), 1])
            for k in range(n):
                assert abs(float(rew[r[k]]) - (cut(s1[k]) - cut(s0[k])) / deg) <= 1e-6


@pytest.mark.parametrize("greedy", [False, True])
def test_s2v_captured_acting_step_fills_the_replay_consistently(tmp_path, greedy):
    """n_envs > 1: the captured acting step with the masked exploration kernel, eps = 1 (before training) and eps = 0
    (greedy from the second step on): s' row 0 is s row 0 with exactly the chosen vertex set to +1, the reward is the dense
    reward, done only on the last step, N distinct actions per episode; greedy actions are the masked argmax of Q."""
    n, E = 20, 4
    kw = dict(initial_exploration_rate=0.0, final_exploration_rate=0.0, replay_start_size=E, minibatch_size=4,
              update_frequency=10 ** 9, update_target_frequency=10 ** 9) if greedy else dict(replay_start_size=10 ** 6)
    agent = make_s2v_agent(tmp_path, er20(), n, n_envs=E, replay_buffer_size=1000, test_frequency=10 ** 9,
                           save_network_frequency=10 ** 9, init_weight_std=0.05, **kw)
    assert agent._act_graph_ok() and agent._episode_steps == n
    agent.learn(timesteps=E * n * 2)
    n_rows = E * n * 2
    assert len(agent.replay_buffer) == n_rows and agent._env.current_step == 0
    _check_episodes(agent, n_rows, n, E)
    if greedy:
        rb = agent.replay_buffer
        for t in range(1, 2 * n):                                            # step 0 came before training was ready
            r = torch.arange(t * E, (t + 1) * E, device=agent.device)
            pred = agent.predict((rb.xn[r], rb.xg[r], rb.graph[r]))
            assert torch.equal(pred.long().cpu(), rb.action[r].cpu())


def test_s2v_one_environment_eager_path(tmp_path):
    """One environment: host draws in the reference's order, actions always among the spins still at -1, the run is
    reproducible from `seed`; max_steps > N still restarts when every spin is flipped."""
    n = 20
    runs = []
    for k in range(2):
        agent = make_s2v_agent(tmp_path / str(k), er20(), 2 * n, n_envs=1, replay_start_size=30, minibatch_size=8,
                               update_frequency=4, test_frequency=10 ** 9, save_network_frequency=10 ** 9,
                               init_weight_std=0.05, final_exploration_step=60, final_exploration_rate=0.2, seed=17)
        assert agent._episode_steps == n
        losses = agent.learn(timesteps=3 * n)
        assert losses and all(np.isfinite(l) for _, l in losses)
        _check_episodes(agent, 3 * n, n, 1)
        runs.append((agent.replay_buffer.action[:3 * n].cpu(), [p.detach().cpu() for p in agent._qnet.parameters()]))
    assert torch.equal(runs[0][0], runs[1][0])
    assert all(torch.equal(a, b) for a, b in zip(runs[0][1], runs[1][1]))


def test_s2v_learn_runs_and_checkpoints(tmp_path):
    """learn() end to end: finite losses, checkpoints with exactly the networks/s2v keys and shapes that load into
    MPNN(n_obs_in=1), test_network with the S2V environment arguments on the saved network, evaluate_agent finite and at most
    the optimal cuts; the shadow's padded columns are still exactly 0.0."""
    from eco_dqn_b200.networks.mpnn import MPNN
    from eco_dqn_b200.experiments.utils import test_network
    from oracle.mpnn import KEYS
    gsz = np.load(os.path.join(GOLDEN, "graphsets.npz"))
    graphs = er20()
    agent = make_s2v_agent(tmp_path, graphs, 20, n_envs=8, update_frequency=8, update_target_frequency=160,
                           replay_start_size=160, replay_buffer_size=1000, test_frequency=320, test_episodes=6,
                           save_network_frequency=480, init_weight_std=0.01, final_exploration_step=600,
                           final_exploration_rate=0.05, weight_decay=1e-3)
    losses = agent.learn(timesteps=8 * 20 * 3)
    assert len(losses) == (480 - 160) // 8 and all(np.isfinite(l) for _, l in losses)
    assert padded_cols_zero(agent._qnet)
    for path in (tmp_path / "net_best.pth", tmp_path / "net480.pth"):
        sd = torch.load(str(path), map_location="cpu")
        assert tuple(sd.keys()) == KEYS
        assert tuple(sd[KEYS[0]].shape) == (64, 1) and tuple(sd[KEYS[1]].shape) == (63, 2)
        assert all(v.is_contiguous() for v in sd.values())
    sd = torch.load(str(tmp_path / "net480.pth"), map_location="cpu")
    for k, v in agent.network.state_dict().items():
        assert torch.equal(sd[k], v.cpu())
    net = MPNN(n_obs_in=1, n_layers=3, n_features=64, n_hid_readout=[], tied_weights=False)
    net.load_state_dict(sd)
    res = test_network(net.cuda().eval(), s2v_env_args(), [g.astype(np.float64) for g in graphs[:2]], "cuda", 1, n_attempts=1)
    assert all(np.isfinite(res["cut"])) and (np.asarray(res["cut"]) <= gsz["er20_opt"][:2]).all()
    score, sol = agent.evaluate_agent()
    assert np.isfinite(score) and 0 < sol <= gsz["er20_opt"][:6].max()
    # a fresh agent loads the checkpoint into what the kernels read
    other = make_s2v_agent(tmp_path / "o", graphs, 20, n_envs=2, init_network_params=str(tmp_path / "net480.pth"))
    for a, b in zip(other._qnet.parameters(), agent._qnet.parameters()):
        assert torch.equal(a, b)


def test_s2v_autograd_route_matches_kernel_route(tmp_path):
    """A loss callable takes autograd through MPNN(n_obs_in=1) on [B, 1 + N, N]; over a few updates its losses and parameters
    stay within tolerance of the kernel route.  (Both act eagerly -- a loss callable has no captured acting step, whose
    warm-up run draws from the agent's generator -- so that both replays hold the same transitions.)"""
    agents = []
    for loss in ("mse", lambda a, b, reduction="mean": F.mse_loss(a, b, reduction=reduction)):
        ag = make_s2v_agent(tmp_path, er20(), 20, n_envs=4, init_weight_std=0.05, replay_start_size=64, loss=loss,
                            initial_learning_rate=1e-5, cuda_graph=False)
        _fill_replay(ag, 160)
        agents.append(ag)
    assert agents[1]._loss_kind is None
    assert torch.equal(agents[0].replay_buffer.xn, agents[1].replay_buffer.xn)
    p0 = [p.detach().clone() for p in agents[0]._qnet.parameters()]
    gen = torch.Generator(device="cuda").manual_seed(9)
    for _ in range(4):
        idx = agents[0].replay_buffer.sample_indices(16, gen)
        la, lb = [float(ag.train_step(ag.replay_buffer.gather(idx))) for ag in agents]
        assert abs(la - lb) <= 1e-4 * abs(lb) + 1e-7, (la, lb)
    for a, b, c in zip(agents[0]._qnet.parameters(), agents[1]._qnet.parameters(), p0):
        assert float((a - b).norm()) <= 0.05 * float((a - c).norm()) + 1e-9
    assert padded_cols_zero(agents[1]._qnet)


def test_s2v_peer_adam_one_rank_equals_device_adam(tmp_path):
    """dp_mode "peer" with one rank: eco_dp_adam on an S2V agent's update equals eco_mpnn_adam_dev bit for bit."""
    agents = [make_s2v_agent(tmp_path / str(k), er20(), 20, n_envs=4, init_weight_std=0.05, replay_start_size=64,
                             weight_decay=0.01) for k in range(2)]
    for ag in agents:
        _fill_replay(ag, 160)
    agents[1].optimizer.attach_peers(1, 0, lambda mine: mine.reshape(1, 64))
    gen = torch.Generator(device="cuda").manual_seed(4)
    for _ in range(4):
        idx = agents[0].replay_buffer.sample_indices(16, gen)
        for ag in agents:
            ag._update(ag.replay_buffer.gather(idx))
        for a, b in zip(agents[0]._qnet.parameters(), agents[1]._qnet.parameters()):
            assert torch.equal(a, b)
    assert agents[1].optimizer.steps == 4 and int(agents[1].optimizer.err_dev.item()) == 0
    assert padded_cols_zero(agents[1]._qnet)
    agents[1].optimizer.close()


def test_s2v_configuration_checks(tmp_path):
    """Irreversible spins train in the S2V-DQN configuration only, with an MPNN(n_obs_in=1)."""
    import eco_dqn_b200.envs.core as ising_env
    from eco_dqn_b200.envs.utils import SetGraphGenerator, RewardSignal
    from eco_dqn_b200.networks.mpnn import MPNN
    from eco_dqn_b200.agents.dqn.dqn import DQN
    gg = SetGraphGenerator([g.astype(np.float64) for g in er20(2)], ordered=True)
    with pytest.raises(NotImplementedError):
        DQN([ising_env.make("SpinSystem", gg, 20, **s2v_env_args())], lambda: MPNN(), n_envs=2, replay_buffer_size=100)
    bad = dict(s2v_env_args(), reward_signal=RewardSignal.BLS)
    with pytest.raises(NotImplementedError):
        DQN([ising_env.make("SpinSystem", gg, 20, **bad)], lambda: MPNN(n_obs_in=1), n_envs=2, replay_buffer_size=100)
