"""Batched rollout engine: torch owns device memory and streams, libecodqn_b200.so does the work.

Host-side mirror of the reference's environment/agent surface for the rollout hot path (SURVEY.md section 8b):

  GraphSet             <- SingleGraphGenerator / SetGraphGenerator payloads (src/envs/utils.py:319-382) +
                          MaximumCutUnbiasedScorer constants (src/envs/score_solver.py:347-375)
  WeightedGraphSet     <- the same for real-valued couplings (EdgeType.RANDOM): fp64 environment, fp32(J) MPNN
  SparseGraphSet       <- the same for integer couplings stored as CSR, up to 32 768 vertices (GSet G55 and up)
  BatchedSpinSystem    <- B x SpinSystemBase (src/envs/spinsystem.py:50-607): reset / step / observation /
                          best_* trackers, struct-of-arrays on the device
  MPNNWeights          <- MPNN.state_dict() (src/networks/mpnn.py:5-32; SURVEY.md appendix A.3)
  BatchedSpinSystem.rollout <- the hot loop of __test_network_batched (experiments/utils.py:169-207)
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import Graphs, Env, Mpnn, SGraphs, WGraphs, WEnv, check, lib

STATE_DICT_KEYS = (
    "node_init_embedding_layer.0.weight",
    "edge_embedding_layer.edge_embedding_NN.weight",
    "edge_embedding_layer.edge_feature_NN.weight",
    "update_node_embedding_layer.0.message_layer.weight",
    "update_node_embedding_layer.0.update_layer.weight",
    "update_node_embedding_layer.1.message_layer.weight",
    "update_node_embedding_layer.1.update_layer.weight",
    "update_node_embedding_layer.2.message_layer.weight",
    "update_node_embedding_layer.2.update_layer.weight",
    "readout_layer.layer_pooled.weight",
    "readout_layer.layers_readout.0.weight",
    "readout_layer.layers_readout.0.bias",
)
STATE_DICT_SHAPES = ((64, 7), (63, 8), (64, 64), (64, 128), (64, 128), (64, 128), (64, 128), (64, 128), (64, 128),
                     (64, 64), (1, 128), (1,))

EPISODE_DTYPE = np.dtype([("step", "<i4"), ("cut", "<i4"), ("best_cut", "<i4"), ("dist", "<i4"),
                          ("n_improving", "<i4"), ("flags", "<i4"), ("n_visited", "<i4"), ("reserved", "<i4"),
                          ("score", "<f8"), ("nscore", "<f8"), ("best_score", "<f8"), ("best_nscore", "<f8"),
                          ("key", "<u8", (2,)), ("total_reward", "<f8"), ("last_reward", "<f8")])
assert EPISODE_DTYPE.itemsize == 96
# BatchedSpinSystem.episodes() of a weighted set: the cut fields are the fp64 cut / best cut of eco_wenv_t
WEIGHTED_EPISODE_DTYPE = np.dtype([(n, "<f8" if n in ("cut", "best_cut") else EPISODE_DTYPE.fields[n][0])
                                   for n in EPISODE_DTYPE.names])


def _require_cuda(device=None):
    if not torch.cuda.is_available():
        raise RuntimeError("eco_dqn_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("eco_dqn_b200 runs on CUDA devices only (got %s)" % dev)
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _view(ws, ptr, count, dtype, shape):
    off = ptr - ws.data_ptr()
    nbytes = count * torch.empty((), dtype=dtype).element_size()
    return ws[off:off + nbytes].view(dtype).view(*shape)


def time_since_flip_table(T):
    """k-fold fp64 accumulation of 1/T from 0, as `state[idx,:] += 1./max_steps` does (spinsystem.py:493)."""
    t = np.zeros(T + 1, dtype=np.float64)
    acc, inc = 0.0, 1.0 / T
    for k in range(1, T + 1):
        acc = acc + inc
        t[k] = acc
    return t


def immanency_table(T, horizon=None):
    """max(0, ((step - max_steps) / horizon) + 1) per step (spinsystem.py:509-511); entry 0 is the reset value."""
    horizon = T if horizon is None else horizon
    t = np.zeros(T + 1, dtype=np.float64)
    for k in range(1, T + 1):
        t[k] = max(0, ((k - T) / horizon) + 1)
    return t


def zobrist_keys(n_padded, seed=0x5EC0D0):
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.integers(0, 2 ** 64, size=(n_padded, 2), dtype=np.uint64)


def graphs_to_int8(graphs):
    """list / array of dense symmetric adjacency matrices -> int8 [G, N, N].  Real-valued couplings
    (EdgeType.RANDOM) are outside the accelerated path."""
    arr = np.asarray(graphs)
    if arr.ndim == 2:
        arr = arr[None]
    if arr.ndim != 3 or arr.shape[1] != arr.shape[2]:
        raise ValueError("graphs must be [G, N, N] (all graphs of one set share N), got shape %s" % (arr.shape,))
    if arr.dtype != np.int8:
        r = np.rint(arr)
        if not np.array_equal(r, arr) or np.abs(r).max(initial=0) > 127:
            raise NotImplementedError("only integer couplings in [-127, 127] are supported (EdgeType.UNIFORM / "
                                      "DISCRETE); real-valued graphs are outside the accelerated path")
        arr = r.astype(np.int8)
    return np.ascontiguousarray(arr)


def is_int8_graph(graphs):
    """True when every coupling is an integer in [-127, 127] (the int8 path takes it; anything else is a weighted graph)."""
    arr = np.asarray(graphs)
    if arr.dtype == np.int8:
        return True
    if arr.size == 0:
        return True
    if not np.issubdtype(arr.dtype, np.number) or not np.isfinite(arr).all():
        return False
    r = np.rint(arr)
    return bool(np.array_equal(r, arr) and np.abs(r).max(initial=0) <= 127)


class GraphSet:
    weighted = False

    def __init__(self, graphs, device=None, validate=True, min_cut=False, _edges=None):
        """min_cut=True: the scorer constants (and every mask the env kernels derive from the graphs) are those of
        OptimisationTarget.MIN_CUT (reference score_solver.py:423-505) instead of CUT.
        (`_edges`: see GraphSet.from_edges -- the graphs arrive as edge lists, no dense matrix on the host.)"""
        self.device = _require_cuda(device)
        self.min_cut = bool(min_cut)
        if _edges is None:
            J = graphs_to_int8(graphs)
            self.G, self.N = int(J.shape[0]), int(J.shape[1])
        else:
            self.G, self.N = len(_edges["offsets"]) - 1, int(_edges["n"])
        if self.N > _lib.MAX_SPINS:
            raise ValueError("N=%d exceeds ECO_MAX_SPINS=%d" % (self.N, _lib.MAX_SPINS))
        L = lib()
        with torch.cuda.device(self.device):
            nbytes = L.eco_graphs_workspace_bytes(self.G, self.N)
            self._ws = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)    # (padding between the arrays stays defined)
            self.c = Graphs()
            check(L.eco_graphs_bind(C.byref(self.c), _ptr(self._ws), self.G, self.N))
            self.c.reserved = _lib.GRAPHS_MIN_CUT if self.min_cut else 0     # read by the prepare kernel
            if _edges is None:
                Jd = torch.from_numpy(J).to(self.device, non_blocking=False)
                check(L.eco_graphs_load_dev(C.byref(self.c), _ptr(Jd), _stream()))
            else:
                dev = {k: torch.from_numpy(np.ascontiguousarray(_edges[k])).to(self.device) for k in ("offsets", "rows", "cols", "w")}
                check(L.eco_graphs_load_edges_dev(C.byref(self.c), 0, self.G, _ptr(dev["offsets"]), _ptr(dev["rows"]), _ptr(dev["cols"]),
                                                  _ptr(dev["w"]), int(_edges["offsets"][-1]), int(_edges["symmetric"]), _stream()))
            self.NP = int(self.c.NP)
            self.J = _view(self._ws, self.c.J, self.G * self.NP * self.NP, torch.int8, (self.G, self.NP, self.NP))
            self.gscal = _view(self._ws, self.c.gscal, self.G * 4, torch.float64, (self.G, 4))
            self.deg = _view(self._ws, self.c.deg, self.G * self.NP, torch.float32, (self.G, self.NP))
            self.gstat = _view(self._ws, self.c.gstat, self.G * 4, torch.int32, (self.G, 4))
            stat = self.gstat.cpu().numpy()
        self.max_degree = int(stat[:, 0].max())
        self.pm1_only = not bool((stat[:, 3] & 1).any())
        # couplings in {-1,0,1} -> tcgen05 MPNN path allowed
        self.c.reserved = (_lib.GRAPHS_PM1 if self.pm1_only else 0) | (_lib.GRAPHS_MIN_CUT if self.min_cut else 0)
        if validate:
            if (stat[:, 3] & 4).any():
                raise ValueError("graph %d is not symmetric with a zero diagonal" % int(np.nonzero(stat[:, 3] & 4)[0][0]))
            if (stat[:, 3] & 2).any():
                # the reference recurses forever on such a graph (spinsystem.py:209-211)
                raise ValueError("graph %d has no non-zero weighted degree" % int(np.nonzero(stat[:, 3] & 2)[0][0]))
            if stat[:, 2].max() > 32767:
                raise NotImplementedError("weighted degree exceeds the int16 local-field range")

    @classmethod
    def from_edges(cls, n_vertices, graphs, device=None, validate=True, min_cut=False):
        """Sparse ingest (C ABI `eco_graphs_load_edges_dev`): `graphs` is a list whose entries are either
        `(rows, cols, weights)` -- every undirected edge once, as `read_mc_instance` returns them (GSet `.mc` files, reference
        experiments/utils.py:395-406) -- or scipy sparse matrices (the csr pickles of :420-432, every stored entry).  Only
        the edge arrays cross PCIe (5 bytes per entry instead of N*N); the dense int8 couplings are built on the device.
        Weights must be integers in [-127, 127]."""
        import scipy.sparse as sps
        offsets, rows, cols, wts, symmetric = [0], [], [], [], None
        for gph in graphs:
            if sps.issparse(gph):
                coo = gph.tocoo()
                if coo.shape != (n_vertices, n_vertices):
                    raise ValueError("sparse matrix of shape %s in a set of %d-vertex graphs" % (coo.shape, n_vertices))
                r, c_, w_, sym = coo.row, coo.col, coo.data, False
            else:
                r, c_, w_ = gph
                sym = True
            if symmetric is None:
                symmetric = sym
            elif symmetric != sym:
                raise ValueError("edge lists and sparse matrices cannot be mixed in one call")
            w_ = np.asarray(w_)
            if w_.size and (np.abs(w_) > 127).any() or (w_ != np.round(w_)).any():
                raise NotImplementedError("couplings must be integers in [-127, 127]")
            rows.append(np.asarray(r, dtype=np.int32)); cols.append(np.asarray(c_, dtype=np.int32)); wts.append(w_.astype(np.int8))
            offsets.append(offsets[-1] + len(w_))
        cat = lambda xs, dt: np.concatenate(xs).astype(dt) if offsets[-1] else np.zeros(1, dtype=dt)
        edges = {"n": n_vertices, "offsets": np.asarray(offsets, dtype=np.int64), "rows": cat(rows, np.int32),
                 "cols": cat(cols, np.int32), "w": cat(wts, np.int8), "symmetric": bool(symmetric)}
        return cls(None, device=device, validate=validate, min_cut=min_cut, _edges=edges)

    @property
    def mlr(self):
        return self.gscal[:, 0]

    @property
    def qn(self):
        return self.gscal[:, 1]

    @property
    def lb(self):
        return self.gscal[:, 2]


class WeightedGraphSet:
    """G dense symmetric graphs with real-valued couplings (EdgeType.RANDOM: 2*rand-1 weights, or any non-integer matrix a
    SingleGraphGenerator / SetGraphGenerator / load_graph_set hands over), shared read-only by all episodes.  The environment
    runs in fp64 on these couplings, as the reference's fp64 `matrix` does; the MPNN reads their fp32 cast, as the
    reference's drivers do with `.float()` (experiments/utils.py:174).  ECO-DQN configuration (CUT target) only."""
    weighted = True
    min_cut = False
    pm1_only = False

    def __init__(self, graphs, device=None, validate=True):
        self.device = _require_cuda(device)
        arr = np.asarray(graphs, dtype=np.float64)
        if arr.ndim == 2:
            arr = arr[None]
        if arr.ndim != 3 or arr.shape[1] != arr.shape[2]:
            raise ValueError("graphs must be [G, N, N] (all graphs of one set share N), got shape %s" % (arr.shape,))
        self.G, self.N = int(arr.shape[0]), int(arr.shape[1])
        if self.N > _lib.MAX_SPINS:
            raise ValueError("N=%d exceeds ECO_MAX_SPINS=%d" % (self.N, _lib.MAX_SPINS))
        if self.G < 1 or self.N < 1:
            raise ValueError("empty graph set")
        L = lib()
        with torch.cuda.device(self.device):
            self._ws = torch.zeros(L.eco_wgraphs_workspace_bytes(self.G, self.N), dtype=torch.uint8, device=self.device)
            self.c = WGraphs()
            check(L.eco_wgraphs_bind(C.byref(self.c), _ptr(self._ws), self.G, self.N))
            Jd = torch.from_numpy(np.ascontiguousarray(arr)).to(self.device)
            check(L.eco_wgraphs_load_dev(C.byref(self.c), _ptr(Jd), _stream()))
            self.NP = int(self.c.NP)
            G, NP = self.G, self.NP
            self.J = _view(self._ws, self.c.J, G * NP * NP, torch.float64, (G, NP, NP))
            self.Jf = _view(self._ws, self.c.Jf, G * NP * NP, torch.float32, (G, NP, NP))
            self.gscal = _view(self._ws, self.c.gscal, G * 4, torch.float64, (G, 4))
            self.deg = _view(self._ws, self.c.deg, G * NP, torch.float32, (G, NP))
            self.gstat = _view(self._ws, self.c.gstat, G * 4, torch.int32, (G, 4))
            stat = self.gstat.cpu().numpy()
        self.max_degree = int(stat[:, 0].max())
        if validate:
            first = lambda bit: int(np.nonzero(stat[:, 3] & bit)[0][0])
            if (stat[:, 3] & _lib.WGRAPH_NONFINITE).any():
                raise ValueError("graph %d has a non-finite coupling" % first(_lib.WGRAPH_NONFINITE))
            if (stat[:, 3] & _lib.WGRAPH_ASYMMETRIC).any():
                raise ValueError("graph %d is not symmetric with a zero diagonal" % first(_lib.WGRAPH_ASYMMETRIC))
            if (stat[:, 3] & _lib.WGRAPH_NO_DEGREE).any():
                # the reference recurses forever on such a graph (spinsystem.py:209-211)
                raise ValueError("graph %d has no non-zero weighted degree" % first(_lib.WGRAPH_NO_DEGREE))

    @property
    def mlr(self):
        return self.gscal[:, 0]

    @property
    def qn(self):
        return self.gscal[:, 1]

    @property
    def lb(self):
        return self.gscal[:, 2]


def sparse_csr(n_vertices, graphs):
    """Host canonicalisation of SparseGraphSet's input -> (row_ptr int64 [G*N + 1], col int32 [nnz], val int8 [nnz]).

    Each entry of `graphs` is a `(rows, cols, weights)` triple -- every undirected edge once, as `read_mc_instance` returns
    them; both directions are stored --, a scipy sparse matrix (every stored entry, as is) or a dense array (its non-zeros).
    Duplicates resolve last-writer-wins, as in `eco_graphs_load_edges_dev` (the reference's `matrix[i, j] = w`); entries
    whose final value is zero are dropped; columns are ascending within every row."""
    import scipy.sparse as sps
    n = int(n_vertices)
    if n < 1 or n > _lib.MAX_SPINS_SPARSE:
        raise ValueError("N=%d outside [1, ECO_MAX_SPINS_SPARSE=%d]" % (n, _lib.MAX_SPINS_SPARSE))
    counts, cols, vals = [], [], []
    for gph in graphs:
        if sps.issparse(gph):
            coo = gph.tocoo()
            if coo.shape != (n, n):
                raise ValueError("sparse matrix of shape %s in a set of %d-vertex graphs" % (coo.shape, n))
            r, c, w = np.asarray(coo.row, dtype=np.int64), np.asarray(coo.col, dtype=np.int64), np.asarray(coo.data)
        elif isinstance(gph, tuple) and len(gph) == 3:
            r0, c0, w0 = (np.asarray(x).ravel() for x in gph)
            if not (len(r0) == len(c0) == len(w0)):
                raise ValueError("rows, cols and weights must have the same length")
            # (i, j, w) then (j, i, w) for every edge, in input order: the later writer of a position wins
            r = np.stack([r0, c0], axis=1).ravel().astype(np.int64)
            c = np.stack([c0, r0], axis=1).ravel().astype(np.int64)
            w = np.repeat(w0, 2)
        else:
            arr = np.asarray(gph)
            if arr.shape != (n, n):
                raise ValueError("dense graph of shape %s in a set of %d-vertex graphs" % (arr.shape, n))
            r, c = np.nonzero(arr)
            w = arr[r, c]
        if w.size and (not np.issubdtype(w.dtype, np.number) or not np.isfinite(w).all() or
                       (np.rint(w) != w).any() or np.abs(w).max() > 127):
            raise NotImplementedError("sparse graph sets take integer couplings in [-127, 127]; real-valued graphs of more "
                                      "than %d vertices are not supported" % _lib.MAX_SPINS)
        if w.size and (r.min() < 0 or c.min() < 0 or r.max() >= n or c.max() >= n):
            raise ValueError("an entry names a vertex outside [0, %d)" % n)
        key = r * n + c
        # last occurrence of every position: first occurrence in the reversed order; np.unique sorts the keys (row, col)
        ukey, first_rev = np.unique(key[::-1], return_index=True)
        uval = w[::-1][first_rev]
        keep = uval != 0
        ukey, uval = ukey[keep], uval[keep]
        counts.append(np.bincount(ukey // n, minlength=n))
        cols.append((ukey % n).astype(np.int32))
        vals.append(np.rint(uval).astype(np.int8))
    if not counts:
        raise ValueError("empty graph set")
    row_ptr = np.zeros(len(counts) * n + 1, dtype=np.int64)
    np.cumsum(np.concatenate(counts), out=row_ptr[1:])
    return row_ptr, np.concatenate(cols), np.concatenate(vals)


class SparseGraphSet:
    """G integer-weight graphs of up to ECO_MAX_SPINS_SPARSE (32 768) vertices stored as CSR on the device: the GSet instances
    (G55 and up) that the dense N x N layout of GraphSet cannot hold.  The host canonicalises the input (sparse_csr) and
    uploads row_ptr / col / val only; the device computes the scorer constants, the degrees and the validity flags.
    ECO-DQN rollout configuration (CUT target) and the Greedy baseline.  Any N >= 1 is accepted (for N <= 2048 every
    result equals GraphSet's)."""
    weighted = False
    sparse = True
    min_cut = False

    def __init__(self, n_vertices, graphs, device=None, validate=True, min_cut=False):
        if min_cut:
            raise NotImplementedError("OptimisationTarget.MIN_CUT is not supported on sparse graph sets (CUT target only)")
        self.device = _require_cuda(device)
        row_ptr, col, val = sparse_csr(n_vertices, graphs)
        self.N = int(n_vertices)
        self.G = (len(row_ptr) - 1) // self.N
        self.nnz = int(row_ptr[-1])
        L = lib()
        with torch.cuda.device(self.device):
            self._ws = torch.zeros(L.eco_sgraphs_workspace_bytes(self.G, self.N, self.nnz), dtype=torch.uint8, device=self.device)
            self.c = SGraphs()
            check(L.eco_sgraphs_bind(C.byref(self.c), _ptr(self._ws), self.G, self.N, self.nnz))
            dev = [torch.from_numpy(np.ascontiguousarray(x)).to(self.device) for x in (row_ptr, col, val)]
            check(L.eco_sgraphs_load_dev(C.byref(self.c), _ptr(dev[0]), _ptr(dev[1]), _ptr(dev[2]), _stream()))
            self.NP = int(self.c.NP)
            G, NP, nnz = self.G, self.NP, self.nnz
            self.row_ptr = _view(self._ws, self.c.row_ptr, G * self.N + 1, torch.int64, (G * self.N + 1,))
            self.col = _view(self._ws, self.c.col, nnz, torch.int32, (nnz,))
            self.val = _view(self._ws, self.c.val, nnz, torch.int8, (nnz,))
            self.gscal = _view(self._ws, self.c.gscal, G * 4, torch.float64, (G, 4))
            self.deg = _view(self._ws, self.c.deg, G * NP, torch.float32, (G, NP))
            self.gstat = _view(self._ws, self.c.gstat, G * 4, torch.int32, (G, 4))
            self.dmax = _view(self._ws, self.c.dmax, 1, torch.float32, (1,))
            stat = self.gstat.cpu().numpy()
        self.max_degree = int(stat[:, 0].max())
        self.pm1_only = not bool((stat[:, 3] & 1).any())
        self.c.reserved = _lib.GRAPHS_PM1 if self.pm1_only else 0
        if validate:
            first = lambda bit: int(np.nonzero(stat[:, 3] & bit)[0][0])
            if (stat[:, 3] & _lib.SGRAPH_NONCANONICAL).any():
                raise ValueError("graph %d is not canonical CSR" % first(_lib.SGRAPH_NONCANONICAL))
            if (stat[:, 3] & 4).any():
                raise ValueError("graph %d is not symmetric with a zero diagonal" % first(4))
            if (stat[:, 3] & 2).any():
                # the reference recurses forever on such a graph (spinsystem.py:209-211)
                raise ValueError("graph %d has no non-zero weighted degree" % first(2))
            if stat[:, 2].max() > 32767:
                raise NotImplementedError("weighted degree exceeds the int16 local-field range")

    @property
    def mlr(self):
        return self.gscal[:, 0]

    @property
    def qn(self):
        return self.gscal[:, 1]

    @property
    def lb(self):
        return self.gscal[:, 2]


def graph_set(graphs, device=None, validate=True, min_cut=False):
    """GraphSet when every coupling is an integer in [-127, 127], WeightedGraphSet otherwise (what the drop-in surface
    routes through: integer graphs keep the int8 path and its results bit for bit)."""
    if is_int8_graph(graphs):
        return GraphSet(graphs, device=device, validate=validate, min_cut=min_cut)
    if min_cut:
        raise NotImplementedError("OptimisationTarget.MIN_CUT with real-valued couplings is not supported "
                                  "(weighted graphs run the CUT target only)")
    return WeightedGraphSet(graphs, device=device, validate=validate)


class MPNNWeights:
    """fp32 device copies of the 12 reference tensors + the C struct pointing at them."""

    def __init__(self, state_dict, device=None, pack=True):
        self.device = _require_cuda(device)
        self.tensors = []
        self.n_obs_in = 7
        self.aliases = True        # every tensor IS the caller's storage (fp32, contiguous, on the device): see repack()
        for i, (k, shp) in enumerate(zip(STATE_DICT_KEYS, STATE_DICT_SHAPES)):
            if k not in state_dict:
                raise KeyError("state_dict is missing %r (expected the reference MPNN layout, n_obs_in=7 or 1, 3 layers, "
                               "64 features, untied, no hidden readout)" % k)
            t = torch.as_tensor(np.asarray(state_dict[k]) if not torch.is_tensor(state_dict[k]) else state_dict[k])
            t = t.detach().to(self.device, torch.float32).contiguous()
            # S2V-DQN networks (n_obs_in = 1: the spin only; shipped under networks/s2v): W_init is [64, 1] and W_e is
            # [63, 2].  The kernels always see 7 observables; zero columns for the other six give the same result.
            if i < 2 and tuple(t.shape) == (shp[0], shp[1] - 6):
                self.n_obs_in = 1
                t = torch.cat([t, torch.zeros(shp[0], 6, dtype=torch.float32, device=self.device)], dim=1).contiguous()
            if tuple(t.shape) != shp:
                raise ValueError("%s has shape %s, expected %s" % (k, tuple(t.shape), shp))
            src = state_dict[k]
            self.aliases = self.aliases and torch.is_tensor(src) and src.data_ptr() == t.data_ptr()
            self.tensors.append(t)
        t = self.tensors
        self.c = Mpnn()
        self.c.w_init, self.c.w_edge, self.c.w_edge_feat = t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr()
        for l in range(3):
            self.c.w_msg[l] = t[3 + 2 * l].data_ptr()
            self.c.w_upd[l] = t[4 + 2 * l].data_ptr()
        self.c.w_pool, self.c.w_read, self.c.b_read = t[9].data_ptr(), t[10].data_ptr(), t[11].data_ptr()
        self.c.packed = None
        self._packed = None
        L = lib()
        nb = L.eco_mpnn_packed_bytes()
        if pack and nb > 0:
            with torch.cuda.device(self.device):
                self._packed = torch.empty(nb, dtype=torch.uint8, device=self.device)
                check(L.eco_mpnn_pack(C.byref(self.c), _ptr(self._packed), _stream()))
            self.c.packed = self._packed.data_ptr()

    def repack(self):
        """The caller changed the weights in place (an optimizer step on aliased storage): rebuild the bf16 hi/lo
        operand copy the tensor-core kernels read; the fp32 pointers are the live parameters already."""
        if self._packed is not None:
            with torch.cuda.device(self.device):
                check(lib().eco_mpnn_pack(C.byref(self.c), _ptr(self._packed), _stream()))

    def state_dict(self):
        return {k: t.clone() for k, t in zip(STATE_DICT_KEYS, self.tensors)}


class BatchedSpinSystem:
    """B independent Max-Cut ECO-DQN episodes on the device (DEFAULT_OBSERVABLES, BLS reward, normalised,
    reversible spins, infinite memory, Stopping.NORMAL -- the configuration every reference script uses)."""

    def __init__(self, graphset, n_envs, max_steps, basin_reward=None, mpnn_impl=_lib.MPNN_AUTO, reversible_spins=True,
                 dense_reward=False):
        """reversible_spins=False, dense_reward=True, basin_reward=None is the S2V-DQN configuration of the reference
        (experiments/pretrained_agent/test_s2v.py): spins start at -1 and are flipped at most once, the reward is the
        normalised score change, the network / greedy policies choose among the spins still at -1."""
        self.gs = graphset
        self.device = graphset.device
        self.B, self.N, self.T = int(n_envs), graphset.N, int(max_steps)
        if self.B < 1:
            raise ValueError("n_envs must be >= 1")
        if not (1 <= self.T <= 65535):
            raise ValueError("max_steps must be in [1, 65535]")
        # real-valued couplings: fp64 fields (eco_wenv_t), ECO-DQN configuration only
        self.weighted = bool(getattr(graphset, "weighted", False))
        if self.weighted and (not reversible_spins or dense_reward):
            raise NotImplementedError("irreversible spins / dense reward (S2V-DQN) with real-valued couplings are not "
                                      "supported: weighted graphs run the ECO-DQN configuration only")
        # CSR graph sets: the int8 state (eco_env_t) stepped in O(degree), ECO-DQN configuration only
        self.sparse = bool(getattr(graphset, "sparse", False))
        if self.sparse and (not reversible_spins or dense_reward):
            raise NotImplementedError("irreversible spins / dense reward (S2V-DQN) are not supported on sparse graph sets: "
                                      "they run the ECO-DQN configuration only")
        self.basin_reward = basin_reward
        self.mpnn_impl = mpnn_impl
        L = lib()
        basin = float(basin_reward) if basin_reward is not None else -1.0
        with torch.cuda.device(self.device):
            if self.weighted:
                nbytes = L.eco_wenv_workspace_bytes(self.B, self.N, self.T)
                self._ws = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
                self.c = WEnv()
                check(L.eco_wenv_bind(C.byref(self.c), _ptr(self._ws), self.B, self.N, self.T, basin))
                self._base = self.c.base        # (shares the memory of self.c)
            elif self.sparse:
                nbytes = L.eco_senv_workspace_bytes(self.B, self.N, self.T)
                self._ws = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
                self.c = Env()
                check(L.eco_senv_bind(C.byref(self.c), _ptr(self._ws), self.B, self.N, self.T, basin))
                self._base = self.c
            else:
                nbytes = L.eco_env_workspace_bytes(self.B, self.N, self.T)
                self._ws = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
                self.c = Env()
                check(L.eco_env_bind(C.byref(self.c), _ptr(self._ws), self.B, self.N, self.T, basin))
                self._base = self.c
            base = self._base
            self.NP, self.NW = int(base.NP), int(base.NW)
            self.reversible_spins, self.dense_reward = bool(reversible_spins), bool(dense_reward)
            base.reserved = (0 if reversible_spins else _lib.ENV_IRREVERSIBLE) | (_lib.ENV_DENSE_REWARD if dense_reward else 0)
            zob = np.ascontiguousarray(zobrist_keys(self.NP))
            tsf = time_since_flip_table(self.T).astype(np.float32)
            imm = immanency_table(self.T).astype(np.float32)
            check(L.eco_env_set_tables(C.byref(base), zob.ctypes.data_as(C.c_void_p), tsf.ctypes.data_as(C.c_void_p),
                                       imm.ctypes.data_as(C.c_void_p), _stream()))
            torch.cuda.current_stream().synchronize()   # host tables are temporaries
            B, NP = self.B, self.NP
            ws = self._ws
            self.spins = _view(ws, base.spins, B * NP, torch.int8, (B, NP))
            if self.weighted:
                self.hfield = _view(ws, self.c.h, B * NP, torch.float64, (B, NP))
                self.cuts = _view(ws, self.c.cut, B * 2, torch.float64, (B, 2))     # current cut, best cut
            else:
                self.hfield = _view(ws, base.hfield, B * NP, torch.int16, (B, NP))
            self.last_flip = _view(ws, base.last_flip, B * NP, torch.int16, (B, NP))
            self.diff_bits = _view(ws, base.diff_bits, B * self.NW, torch.int32, (B, self.NW))
            self.graph_idx = _view(ws, base.graph_idx, B, torch.int32, (B,))
            self._ep = _view(ws, base.ep, B * 96, torch.uint8, (B, 96))
            self.xn = _view(ws, base.xn, B * 3 * NP, torch.float32, (B, 3, NP))
            self.xg = _view(ws, base.xg, B * 4, torch.float32, (B, 4))
            self._actions = torch.zeros(B, dtype=torch.int32, device=self.device)
            self._reward = torch.zeros(B, dtype=torch.float64, device=self.device)
            self._done = torch.zeros(B, dtype=torch.uint8, device=self.device)
            self._scratch = None
        self.current_step = 0
        self._is_reset = False

    # ------------------------------------------------------------------ reset / step
    def reset(self, spins=None, graph_idx=None):
        """reference spinsystem.py:183-259.  spins: [B, N] in {-1,+1} (None: 2*randint(2)-1 per episode from the
        global numpy RNG, like spinsystem.py:294).  graph_idx: [B] (None: episode b uses graph b % G)."""
        B, N = self.B, self.N
        if spins is None:
            if self.reversible_spins:
                spins = np.stack([2 * np.random.randint(2, size=N) - 1 for _ in range(B)])
            else:
                spins = -np.ones((B, N), dtype=np.int8)        # spinsystem.py:296-297: irreversible spins start at -1
        if torch.is_tensor(spins):
            sp = spins.to(self.device)
            if sp.shape != (B, N):
                raise ValueError("spins must be [B=%d, N=%d], got %s" % (B, N, tuple(sp.shape)))
            if not bool(((sp == 1) | (sp == -1)).all()):
                raise Exception("SpinSystem is configured for signed spins ([-1,1]).")   # spinsystem.py:604-606
            sp = sp.to(torch.int8).contiguous()
        else:
            spins = np.asarray(spins)
            if spins.shape != (B, N):
                raise ValueError("spins must be [B=%d, N=%d], got %s" % (B, N, spins.shape))
            if not np.isin(spins, [-1, 1]).all():
                raise Exception("SpinSystem is configured for signed spins ([-1,1]).")
            sp = torch.from_numpy(np.ascontiguousarray(spins.astype(np.int8))).to(self.device)
        if graph_idx is None:
            gi = torch.arange(B, dtype=torch.int32, device=self.device) % self.gs.G
        else:
            gi = torch.as_tensor(graph_idx).to(self.device, torch.int32).contiguous()
            if gi.shape != (B,):
                raise ValueError("graph_idx must be [B]")
            if int(gi.min()) < 0 or int(gi.max()) >= self.gs.G:
                raise ValueError("graph_idx out of range")
        with torch.cuda.device(self.device):
            reset = lib().eco_wenv_reset if self.weighted else lib().eco_senv_reset if self.sparse else lib().eco_env_reset
            check(reset(C.byref(self.gs.c), C.byref(self.c), _ptr(gi), _ptr(sp), _stream()))
        self.current_step = 0
        self._is_reset = True
        return self

    def _check_steppable(self, n=1):
        if not self._is_reset:
            raise RuntimeError("call reset() before step()")
        if self.current_step + n > self.T:
            # reference: "The environment has already returned done. Stop it!" (spinsystem.py:365-367)
            raise NotImplementedError("The environment has already returned done. Stop it!")

    def step(self, actions, hist=None):
        """reference spinsystem.py:355-559 for all B episodes.  Returns (reward fp64 [B], done uint8 [B])."""
        self._check_steppable()
        a = torch.as_tensor(actions).to(self.device, torch.int32).contiguous()
        if a.shape != (self.B,):
            raise ValueError("actions must be [B]")
        ha, hr, hs = hist if hist is not None else (None, None, None)
        step = self._step_fn()
        with torch.cuda.device(self.device):
            check(step(C.byref(self.gs.c), C.byref(self.c), _lib.POLICY_ACTIONS, _ptr(a),
                                     _ptr(self._reward), _ptr(self._done), _ptr(ha), _ptr(hr), _ptr(hs), _stream()))
        self.current_step += 1
        return self._reward, self._done

    def _step_fn(self):
        return lib().eco_wenv_step if self.weighted else lib().eco_senv_step if self.sparse else lib().eco_env_step

    def greedy_step(self, hist=None):
        """One step of the Greedy solver (src/agents/solver.py:105-131) for every episode still running."""
        self._check_steppable()
        ha, hr, hs = hist if hist is not None else (None, None, None)
        step = self._step_fn()
        with torch.cuda.device(self.device):
            check(step(C.byref(self.gs.c), C.byref(self.c), _lib.POLICY_GREEDY, None,
                                     _ptr(self._reward), _ptr(self._done), _ptr(ha), _ptr(hr), _ptr(hs), _stream()))
        self.current_step += 1
        return self._reward, self._done

    # ------------------------------------------------------------------ Q-network
    def _scratch_for(self, B):
        if self.sparse:
            nb = lib().eco_smpnn_scratch_bytes(B, self.N)
        else:
            nb = lib().eco_mpnn_scratch_bytes(B, self.N, self.mpnn_impl)
        if self._scratch is None or self._scratch.numel() < nb:
            self._scratch = torch.empty(nb, dtype=torch.uint8, device=self.device)
        return self._scratch

    def _sparse_impl(self, weights, impl):
        """The Q-network of a CSR set: AUTO / SIMT run the gather forward with fp32 linears (eco_smpnn_forward), TCGEN05
        its per-vertex linears on the tensor cores (eco_smpnn_forward_impl), which read the packed bf16 hi/lo weights."""
        use = self.mpnn_impl if impl is None else impl
        if use == _lib.MPNN_TCGEN05 and weights is not None and weights._packed is None:
            raise ValueError("the tensor-core Q-network needs packed weights: MPNNWeights(..., pack=True)")
        return use

    def q_values(self, weights, norm_max=None, want_actions=True, impl=None):
        """MPNN.forward on the current observations (mpnn.py:40-77) -> (Q fp32 [B, N], argmax int32 [B])."""
        q = torch.zeros(self.B, self.NP, dtype=torch.float32, device=self.device)
        acts = self._actions if want_actions else None
        nm = float(norm_max) if norm_max is not None else 0.0
        if self.sparse:
            use = self._sparse_impl(weights, impl)
            with torch.cuda.device(self.device):
                if use == _lib.MPNN_TCGEN05:
                    check(lib().eco_smpnn_forward_impl(C.byref(self.gs.c), C.byref(weights.c), self.B, _ptr(self.graph_idx),
                                                       _ptr(self.xn), _ptr(self.xg), nm, _ptr(q), _ptr(acts),
                                                       _ptr(self._scratch_for(self.B)), use, _stream()))
                else:
                    check(lib().eco_smpnn_forward(C.byref(self.gs.c), C.byref(weights.c), self.B, _ptr(self.graph_idx),
                                                  _ptr(self.xn), _ptr(self.xg), nm, _ptr(q), _ptr(acts),
                                                  _ptr(self._scratch_for(self.B)), _stream()))
            return q[:, :self.N], acts
        forward = lib().eco_wmpnn_forward if self.weighted else lib().eco_mpnn_forward
        with torch.cuda.device(self.device):
            check(forward(C.byref(self.gs.c), C.byref(weights.c), self.B, _ptr(self.graph_idx),
                                         _ptr(self.xn), _ptr(self.xg), nm, _ptr(q), _ptr(acts),
                                         _ptr(self._scratch_for(self.B)), self.mpnn_impl if impl is None else impl,
                                         _stream()))
        if acts is not None and not self.reversible_spins:
            # irreversible spins: argmax over the spins still at -1 (experiments/utils.py:67-74)
            with torch.cuda.device(self.device):
                check(lib().eco_env_masked_argmax(C.byref(self.c), _ptr(q), _ptr(acts), _stream()))
        return q[:, :self.N], acts

    def rollout(self, weights=None, n_steps=None, policy="network", norm_max=None, record_history=False, impl=None):
        """n_steps x [Q-eval + argmax -> step] without host round trips (experiments/utils.py:169-207), or the
        Greedy baseline with policy="greedy" (experiments/utils.py:218-227).

        norm_max: the divisor of the degree feature (`norm / norm.max()`, mpnn.py:102).  None (default): every episode
        is normalised by its OWN graph's max degree -- what the reference computes, because __test_network_batched
        batches the attempts of one graph at a time.  0: the max degree over the whole graph set; > 0: that value."""
        n_steps = self.T - self.current_step if n_steps is None else int(n_steps)
        self._check_steppable(n_steps)
        pol = {"network": _lib.POLICY_NETWORK, "greedy": _lib.POLICY_GREEDY}[policy]
        hist = (None, None, None)
        if record_history:
            hist = (torch.full((self.B, self.T), -1, dtype=torch.int32, device=self.device),
                    torch.zeros(self.B, self.T, dtype=torch.float64, device=self.device),
                    torch.zeros(self.B, self.T, dtype=torch.float64, device=self.device))
        if pol == _lib.POLICY_NETWORK and weights is None:
            raise ValueError("network policy needs weights")
        nm = float(norm_max) if norm_max is not None else -1.0
        if self.sparse:
            use = self._sparse_impl(weights, impl) if pol == _lib.POLICY_NETWORK else _lib.MPNN_AUTO
            with torch.cuda.device(self.device):
                if use == _lib.MPNN_TCGEN05:
                    check(lib().eco_srollout_impl(C.byref(self.gs.c), C.byref(self.c), C.byref(weights.c), n_steps, pol, nm,
                                                  _ptr(self._actions), _ptr(self._scratch_for(self.B)), use,
                                                  _ptr(hist[0]), _ptr(hist[1]), _ptr(hist[2]), _stream()))
                else:
                    check(lib().eco_srollout(C.byref(self.gs.c), C.byref(self.c),
                                             C.byref(weights.c) if weights is not None else None, n_steps, pol, nm,
                                             _ptr(self._actions),
                                             _ptr(self._scratch_for(self.B)) if pol == _lib.POLICY_NETWORK else None,
                                             _ptr(hist[0]), _ptr(hist[1]), _ptr(hist[2]), _stream()))
            self.current_step += n_steps
            return hist if record_history else None
        rollout = lib().eco_wrollout if self.weighted else lib().eco_rollout
        with torch.cuda.device(self.device):
            check(rollout(C.byref(self.gs.c), C.byref(self.c),
                                    C.byref(weights.c) if weights is not None else None, n_steps, pol, nm,
                                    _ptr(self._actions),
                                    _ptr(self._scratch_for(self.B)) if pol == _lib.POLICY_NETWORK else None,
                                    self.mpnn_impl if impl is None else impl, _ptr(hist[0]), _ptr(hist[1]),
                                    _ptr(hist[2]), _stream()))
        self.current_step += n_steps
        return hist if record_history else None

    # ------------------------------------------------------------------ views
    def observation(self):
        """Rows 0..6 of get_observation() cast to fp32 (spinsystem.py:561-574; experiments/utils.py:174): [B, 7, N].
        The adjacency rows 7.. are the (static) graph and are never materialised per step."""
        obs = torch.empty(self.B, 7, self.N, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib().eco_env_observation(C.byref(self._base), _ptr(obs), _stream()))
        return obs

    def episodes(self):
        """Per-episode scalar blocks as a numpy structured array (synchronises).  Weighted sets: `cut` / `best_cut` are
        the fp64 values."""
        ep = self._ep.cpu().numpy().view(EPISODE_DTYPE).reshape(self.B)
        if not self.weighted:
            return ep
        out = np.zeros(self.B, dtype=WEIGHTED_EPISODE_DTYPE)
        for n in EPISODE_DTYPE.names:
            out[n] = ep[n]
        cuts = self.cuts.cpu().numpy()
        out["cut"], out["best_cut"] = cuts[:, 0], cuts[:, 1]
        return out

    def results(self):
        """(best_cut int32 [B] -- fp64 for a weighted set --, best_spins int8 [B, N], steps int32 [B]) device tensors."""
        bc = torch.empty(self.B, dtype=torch.float64 if self.weighted else torch.int32, device=self.device)
        bs = torch.empty(self.B, self.N, dtype=torch.int8, device=self.device)
        st = torch.empty(self.B, dtype=torch.int32, device=self.device)
        results = lib().eco_wenv_results if self.weighted else lib().eco_env_results
        with torch.cuda.device(self.device):
            check(results(C.byref(self.c), _ptr(bc), _ptr(bs), _ptr(st), _stream()))
        return bc, bs, st


class HostSession:
    """eco_session_*: the whole batched test_network job behind HOST buffers (the e2e entry point)."""

    def __init__(self, G, N, B, T, basin_reward, state_dict, impl=_lib.MPNN_AUTO):
        _require_cuda()
        if N > _lib.MAX_SPINS:
            raise NotImplementedError("HostSession takes the dense layout (N <= %d); larger graphs run through SparseGraphSet + "
                                      "BatchedSpinSystem" % _lib.MAX_SPINS)
        self.G, self.N, self.B, self.T = G, N, B, T
        self._w = [np.ascontiguousarray(np.asarray(state_dict[k].cpu() if torch.is_tensor(state_dict[k])
                                                   else state_dict[k], dtype=np.float32)) for k in STATE_DICT_KEYS]
        arr = (C.c_void_p * 12)(*[w.ctypes.data for w in self._w])
        self._h = C.c_void_p()
        check(lib().eco_session_create(C.byref(self._h), G, N, B, T,
                                       float(basin_reward) if basin_reward is not None else -1.0, arr, impl))

    def rollout(self, J_host, graph_idx_host, init_spins_host, best_cut_out, best_spins_out=None, policy="network",
                norm_max=None):
        """All arguments are HOST arrays/tensors (pinned recommended); synchronises the current stream.
        norm_max as in BatchedSpinSystem.rollout (None: per-episode graph, like the reference's per-graph batches)."""
        def hp(x):
            if x is None:
                return C.c_void_p(0)
            return C.c_void_p(x.data_ptr()) if torch.is_tensor(x) else x.ctypes.data_as(C.c_void_p)
        if J_host is not None and not is_int8_graph(J_host.cpu().numpy() if torch.is_tensor(J_host) else J_host):
            raise NotImplementedError("HostSession takes int8 couplings only; real-valued graphs run through "
                                      "WeightedGraphSet + BatchedSpinSystem")
        pol = {"network": _lib.POLICY_NETWORK, "greedy": _lib.POLICY_GREEDY}[policy]
        check(lib().eco_session_rollout(self._h, hp(J_host), hp(graph_idx_host), hp(init_spins_host), pol,
                                        float(norm_max) if norm_max is not None else -1.0, hp(best_cut_out),
                                        hp(best_spins_out), _stream()))

    def close(self):
        if self._h:
            lib().eco_session_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
