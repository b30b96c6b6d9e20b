"""Drop-in for reference experiments/utils.py on the rollout path: `test_network` (the batched greedy-Q driver plus
the Greedy baselines) and the graph loaders.  Same signature, same DataFrame columns, same consumption of the
global numpy RNG for the random initial spins -- but every episode of every same-sized graph is stepped on the
device in one batch, with no host round trip per step.

reference experiments/utils.py:22-31 (test_network), :33-303 (__test_network_batched), :391-432 (loaders).
"""
import os
import pickle
import time
from collections import namedtuple

import networkx as nx
import numpy as np
import pandas as pd
import scipy as sp
import torch

from .. import engine
from ..envs.spinsystem import check_supported
from ..envs.utils import DEFAULT_OBSERVABLES, RewardSignal, ExtraAction, OptimisationTarget, SpinBasis, Stopping


def _weights_of(network, device):
    if isinstance(network, engine.MPNNWeights):
        return network
    if hasattr(network, "engine_weights"):
        return network.engine_weights(device)
    if hasattr(network, "state_dict"):
        return engine.MPNNWeights(network.state_dict(), device=device)
    return engine.MPNNWeights(network, device=device)       # a plain dict keyed like the reference's state_dict


def _check_env_args(env_args, n_steps):
    a = dict(observables=DEFAULT_OBSERVABLES, reward_signal=RewardSignal.DENSE, extra_action=ExtraAction.PASS,
             optimisation_target=OptimisationTarget.ENERGY, spin_basis=SpinBasis.SIGNED, norm_rewards=False,
             memory_length=None, horizon_length=None, stag_punishment=None, basin_reward=None, reversible_spins=True,
             init_snap=None, stopping=Stopping.NORMAL)          # SpinSystemFactory.get defaults (spinsystem.py:30-45)
    a.update(env_args)
    check_supported(a["observables"], a["reward_signal"], a["extra_action"], a["optimisation_target"], a["spin_basis"],
                    a["norm_rewards"], a["memory_length"], a["horizon_length"], a["stag_punishment"],
                    a["reversible_spins"], a["init_snap"], a["stopping"], n_steps)
    return a


def test_network(network, env_args, graphs_test, device=None, step_factor=1, batched=True,
                 n_attempts=50, return_raw=False, return_history=False, max_batch_size=None):
    if not batched:
        # the reference's sequential tester calls a method that does not exist (experiments/utils.py:343)
        raise NotImplementedError("only the batched tester is supported (the reference's sequential one is broken)")
    if device is None:
        device = "cuda"
    dev = engine._require_cuda(device)
    weights = _weights_of(network, dev)

    graphs_test = [np.asarray(g) for g in graphs_test]
    n_graphs = len(graphs_test)
    results, results_raw, history = [None] * n_graphs, [None] * n_graphs, [None] * n_graphs
    # irreversible spins (S2V-DQN): every episode starts from all -1, so there is a single attempt per graph and no
    # random-start greedy baseline (experiments/utils.py:87, 218, 253-260); nothing is drawn from the RNG
    reversible = env_args.get('reversible_spins', True)
    if not reversible:
        n_attempts = 1

    # The reference walks the graphs in order and, per graph, draws (1 + n_attempts) x N random spins from numpy's
    # global RNG: N for the constructor's reset (spinsystem.py:168,294), then N per episode (experiments/utils.py:154).
    init = []
    for g in graphs_test:
        n = g.shape[0]
        if reversible:
            np.random.randint(2, size=n)
            init.append(np.stack([2 * np.random.randint(2, size=n) - 1 for _ in range(n_attempts)]).astype(np.int8))
        else:
            init.append(-np.ones((1, n), dtype=np.int8))

    # group graphs of equal size: one graph set, one batch of len(group) x n_attempts episodes
    groups = {}
    for j, g in enumerate(graphs_test):
        groups.setdefault(g.shape[0], []).append(j)
    for n, idxs in groups.items():
        n_steps = int(n * step_factor)
        args = _check_env_args(env_args, n_steps)
        min_cut = args["optimisation_target"] == OptimisationTarget.MIN_CUT
        if n > engine._lib.MAX_SPINS:
            # more vertices than the dense layout holds: integer couplings as CSR (real-valued ones raise)
            gs = engine.SparseGraphSet(n, [graphs_test[j] for j in idxs], device=dev, min_cut=min_cut)
        else:
            # integer couplings in [-127, 127]: the int8 path; anything else (EdgeType.RANDOM): the fp64 weighted path
            gs = engine.graph_set(np.stack([graphs_test[j] for j in idxs]), device=dev, min_cut=min_cut)
        G = len(idxs)
        B = G * n_attempts
        gidx = np.repeat(np.arange(G, dtype=np.int32), n_attempts)
        spins = np.concatenate([init[j] for j in idxs])

        mode = dict(reversible_spins=reversible, dense_reward=args["reward_signal"] == RewardSignal.DENSE)
        env = engine.BatchedSpinSystem(gs, B, n_steps, args["basin_reward"], **mode)
        env.reset(spins=spins, graph_idx=gidx)
        scores0 = env.episodes()["score"].copy() if return_history else None
        torch.cuda.synchronize(dev)
        t_start = time.time()
        hist = env.rollout(weights, record_history=return_history)
        best_cut, best_spins, steps_taken = env.results()
        torch.cuda.synchronize(dev)
        t_total = time.time() - t_start
        steps_taken = steps_taken.cpu().numpy()
        best_cut = best_cut.cpu().numpy().astype(np.float64)
        best_spins = best_spins.cpu().numpy().astype(np.float64)

        # Greedy baselines (experiments/utils.py:100-111, 218-227): from the same random starts, and from all -1
        if reversible:
            env.reset(spins=spins, graph_idx=gidx)
            env.rollout(policy="greedy")
            g_cut, g_spins, _ = env.results()
            g_cut = g_cut.cpu().numpy().astype(np.float64)
            g_spins = g_spins.cpu().numpy().astype(np.float64)
        env1 = engine.BatchedSpinSystem(gs, G, n_steps, args["basin_reward"], **mode)
        env1.reset(spins=-np.ones((G, n), dtype=np.int8), graph_idx=np.arange(G, dtype=np.int32))
        env1.rollout(policy="greedy")
        s_cut, s_spins, _ = env1.results()
        s_cut = s_cut.cpu().numpy().astype(np.float64)
        s_spins = s_spins.cpu().numpy().astype(np.float64)
        if return_history:
            ha, hr, hs = (h.cpu().numpy() for h in hist)

        for k, j in enumerate(idxs):
            sl = slice(k * n_attempts, (k + 1) * n_attempts)
            cuts = best_cut[sl]
            i_best = int(np.argmax(cuts))
            if reversible:
                ig = int(np.argmax(g_cut[sl]))
                gr_cut, gr_spins, gr_mean = g_cut[sl][ig], g_spins[sl][ig], np.mean(g_cut[sl])
                raw_g = [list(g_cut[sl]), list(g_spins[sl])]
            else:                                   # experiments/utils.py:257-260: the single -1 start stands in
                gr_cut, gr_spins, gr_mean = s_cut[k], s_spins[k], s_cut[k]
                raw_g = [[], []]
            results[j] = [cuts[i_best], best_spins[sl][i_best], np.mean(cuts),
                          s_cut[k], s_spins[k],
                          gr_cut, gr_spins, gr_mean,
                          t_total / B]
            results_raw[j] = [[s.astype(np.float64) for s in init[j]], list(cuts), list(best_spins[sl])] + raw_g
            if return_history:
                st = steps_taken[sl]                # an irreversible episode ends once every spin is flipped
                acts = [[None] + [int(a) for a in row[:t]] for row, t in zip(ha[sl], st)]
                rews = [[None] + [float(r) for r in row[:t]] for row, t in zip(hr[sl], st)]
                scs = [[float(s0)] + [float(s) for s in row[:t]] for s0, row, t in zip(scores0[sl], hs[sl], st)]
                history[j] = [acts, scs, rews]
            print('Graph {}, best(mean) cut: {}({}), greedy cut (rand init / +1 init) : {} / {}.  ({} attempts in {}s)'.format(
                j, cuts[i_best], np.mean(cuts), gr_cut, s_cut[k], n_attempts, np.round(t_total * n_attempts / B, 4)))

    results = pd.DataFrame(data=results, columns=["cut", "sol", "mean cut",
                                                  "greedy (+1 init) cut", "greedy (+1 init) sol",
                                                  "greedy (rand init) cut", "greedy (rand init) sol",
                                                  "greedy (rand init) mean cut", "time"])
    results_raw = pd.DataFrame(data=results_raw, columns=["init spins", "cuts", "sols", "greedy cuts", "greedy sols"])
    if return_history:
        history = pd.DataFrame(data=history, columns=["actions", "scores", "rewards"])
    if return_raw == False and return_history == False:
        return results
    ret = [results]
    if return_raw:
        ret.append(results_raw)
    if return_history:
        ret.append(history)
    return ret


Graph = namedtuple('Graph', 'name n_vertices n_edges matrix bk_val bk_sol')      # reference experiments/utils.py:389


def read_mc_instance(path):
    """GSet-style `.mc` text instance -> (n_vertices, n_edges, rows, cols, weights): a header line `n m`, then one
    `i j w` line per edge with 1-based vertex numbers (the format reference experiments/utils.py:395-406 parses).  The edge
    list is kept as arrays so that it can go to the device as int8 dense or as CSR without a dense float64 detour."""
    with open(path) as f:
        header = f.readline().split()
        if len(header) != 2:
            raise AssertionError('First line in file should define graph dimensions.')      # the reference's assert text
        n_vertices, n_edges = int(header[0]), int(header[1])
        body = np.loadtxt(f, dtype=np.int64, ndmin=2) if n_edges > 0 else np.zeros((0, 3), dtype=np.int64)
    if body.shape[1] != 3:
        raise ValueError("%s: edge lines must be `i j w`" % path)
    return n_vertices, n_edges, body[:, 0] - 1, body[:, 1] - 1, body[:, 2]


def load_graph(graph_dir, graph_name):
    """Same result as reference experiments/utils.py:391-418: the instance as a dense symmetric float matrix, the best-known
    value (`bkvl/<name>.bkvl`) and solution (`bksol/<name>.bksol`: one 0/1 character per vertex, to which the reference
    appends one random bit drawn with `np.random.choice([0, 1])` -- kept, it consumes the global RNG)."""
    n_vertices, n_edges, rows, cols, weights = read_mc_instance(os.path.join(graph_dir, 'instances', graph_name + '.mc'))
    matrix = np.zeros((n_vertices, n_vertices))
    matrix[rows, cols] = weights
    matrix[cols, rows] = weights
    with open(os.path.join(graph_dir, 'bkvl', graph_name + '.bkvl')) as f:
        bk_val = float(f.readline())
    with open(os.path.join(graph_dir, 'bksol', graph_name + '.bksol')) as f:
        digits = np.frombuffer(f.readline().strip().encode('ascii'), dtype=np.uint8) - ord('0')
    bk_sol = np.append(digits.astype(np.int64), np.random.choice([0, 1]))
    return Graph(graph_name, n_vertices, n_edges, matrix, bk_val, bk_sol)


def to_dense_adjacency(g):
    """One entry of a pickled graph set -- ndarray, networkx graph (edge attribute `weight`) or any scipy sparse matrix --
    as a dense array, which is what every caller of the reference's loader receives (experiments/utils.py:424-430)."""
    if isinstance(g, nx.Graph):
        return nx.to_numpy_array(g)
    if sp.sparse.issparse(g):
        return g.toarray()
    return g


def load_graph_set(graph_save_loc):
    """Pickled list of graphs -> list of dense arrays (reference experiments/utils.py:420-432)."""
    with open(graph_save_loc, 'rb') as f:
        graphs_test = [to_dense_adjacency(g) for g in pickle.load(f)]
    print('{} target graphs loaded from {}'.format(len(graphs_test), graph_save_loc))
    return graphs_test


def _n_of(g):
    return g.number_of_nodes() if isinstance(g, nx.Graph) else g.shape[0]


def _sparse_adjacency(g):
    """One pickled graph for SparseGraphSet without an N x N host matrix: scipy matrices as they are, networkx graphs through
    their sparse adjacency (the entries of `nx.to_numpy_array`: edge attribute `weight`, default 1, same vertex order),
    anything else as its dense array."""
    if isinstance(g, nx.Graph):
        return nx.to_scipy_sparse_array(g, weight="weight", format="coo")
    return g


def load_graph_set_device(graph_save_loc, device=None, min_cut=False):
    """The same pickle straight into an engine.GraphSet (all graphs of the file must share N, as the reference's batched
    tester assumes per graph anyway).  A file of scipy sparse matrices (the csr pickles) goes through the sparse ingest --
    only the stored entries cross PCIe, the dense int8 couplings are built on the device; anything else is uploaded as int8,
    or, when a coupling is not an integer in [-127, 127], as an fp64 engine.WeightedGraphSet.  Graphs of more than 2048
    vertices become an engine.SparseGraphSet (CSR on the device)."""
    with open(graph_save_loc, 'rb') as f:
        raw = pickle.load(f)
    if len(raw) and _n_of(raw[0]) > engine._lib.MAX_SPINS:
        if min_cut:
            raise NotImplementedError("OptimisationTarget.MIN_CUT is not supported on sparse graph sets (CUT target only)")
        n = _n_of(raw[0])
        return engine.SparseGraphSet(n, [_sparse_adjacency(g) for g in raw], device=device)
    if len(raw) and all(sp.sparse.issparse(g) for g in raw):
        return engine.GraphSet.from_edges(raw[0].shape[0], raw, device=device, min_cut=min_cut)
    graphs = [to_dense_adjacency(g) for g in raw]
    return engine.graph_set(np.stack(graphs), device=device, min_cut=min_cut)


def load_mc_instances_device(graph_dir, graph_names, device=None, min_cut=False):
    """GSet `.mc` instances (all of one size) straight into an engine.GraphSet through the sparse ingest: the edge lists go to
    the device (5 bytes per edge) and the dense int8 couplings are built there -- no N x N float64 matrix, which is what
    `load_graph` (reference experiments/utils.py:391-418) builds per instance.  Instances of more than 2048 vertices (G55 and
    up) become an engine.SparseGraphSet: the same edge lists, kept as CSR on the device."""
    insts = [read_mc_instance(os.path.join(graph_dir, 'instances', name + '.mc')) for name in graph_names]
    n = insts[0][0]
    if any(i[0] != n for i in insts):
        raise ValueError("all instances of one GraphSet must have the same number of vertices")
    if n > engine._lib.MAX_SPINS:
        return engine.SparseGraphSet(n, [(r, c, w) for _, _, r, c, w in insts], device=device, min_cut=min_cut)
    return engine.GraphSet.from_edges(n, [(r, c, w) for _, _, r, c, w in insts], device=device, min_cut=min_cut)


def mk_dir(export_dir, quite=False):
    os.makedirs(export_dir, exist_ok=True)
