"""Oracle: MPNN Q-network forward in float64 over a CSR graph (TEST INFRASTRUCTURE ONLY, see oracle/__init__.py).

The same network as oracle/mpnn.py (reference src/networks/mpnn.py:40-77), restated for precision tests of the kernels:

  * float64 throughout, so its own round-off (~1e-15) is far below anything a kernel test resolves;
  * the graph is a CSR (row_ptr, col, val) shared by the batch, and the edge stage `ReLU(a_ij * w0 + P_j)`, summed per
    target vertex, never forms the [B, N, N, 63] tensor: for integer couplings it is one sparse 0/1 product per distinct
    value, otherwise it runs over edge chunks -- a complete 2048-vertex graph or a 32 768-vertex star fits in memory;
  * the degrees `deg` and the divisor `norm_max` of the degree feature are explicit arguments, so a caller can pass a
    graph with one entry dropped but the original degrees, or a wrong divisor ("mutants": small, deliberate defects whose
    effect on Q a precision test must be able to see);
  * plain torch ops without in-place updates of leaves: weights given as tensors with requires_grad get fp64 gradients
    through autograd.

Pinned against the golden fp32 Q and oracle.mpnn.mpnn_forward_blocked in tests/test_mpnn64_cpu.py.
"""
import warnings

import numpy as np
import torch

from oracle.mpnn import KEYS

F64 = torch.float64
warnings.filterwarnings("ignore", message="Sparse CSR tensor support is in beta state")


def weights64(w):
    """State dict (numpy or torch, any float dtype) -> float64 torch tensors.  Tensors that require grad stay attached."""
    out = {}
    for k in KEYS:
        v = w[k]
        out[k] = v.to(F64) if torch.is_tensor(v) else torch.as_tensor(np.asarray(v), dtype=F64)
    return out


def csr_from_dense(J):
    """Dense [N, N] couplings -> (row_ptr int64 [N+1], col int64 [nnz], val float64 [nnz]), columns ascending per row.
    Non-zeros of J as given: pass fp32(J) for a weighted graph, whose MPNN reads the fp32 couplings."""
    J = np.asarray(J)
    r, c = np.nonzero(J)
    row_ptr = np.zeros(J.shape[0] + 1, dtype=np.int64)
    np.cumsum(np.bincount(r, minlength=J.shape[0]), out=row_ptr[1:])
    return row_ptr, c.astype(np.int64), J[r, c].astype(np.float64)


def degrees(row_ptr):
    """The network's degree: entries per row, 0 clamped to 1 (mpnn.py:36-37)."""
    d = np.diff(np.asarray(row_ptr)).astype(np.float64)
    d[d == 0] = 1
    return d


def drop_entry(csr, i, k=-1):
    """Mutant: the CSR without entry k (default: the last) of row i.  Only row i loses it; pair it with the ORIGINAL
    degrees to model a kernel that skips one neighbour in its gathers."""
    row_ptr, col, val = csr
    pos = int(row_ptr[i + 1] - 1 if k < 0 else row_ptr[i] + k)
    assert row_ptr[i] <= pos < row_ptr[i + 1]
    rp = row_ptr.copy()
    rp[i + 1:] -= 1
    return rp, np.delete(col, pos), np.delete(val, pos)


def forward64(w, x, csr, deg, norm_max, set_max_degree=None, chunk=1 << 17):
    """Q float64 [B, N] of the episodes x: [B, N, 7] (observation rows 0..6, vertex-major) on one graph.

    csr = (row_ptr, col, val): row i's neighbours j and couplings a_ij; deg: [N] the degree divisor (`norm`);
    norm_max: > 0 that value, 0 `set_max_degree` (the graph set's maximum degree), < 0 max(deg) (this graph's)."""
    W = weights64(w)
    x = torch.as_tensor(x, dtype=F64)
    if x.dim() == 2:
        x = x.unsqueeze(0)
    B, N, _ = x.shape
    row_ptr, col, val = csr
    counts = torch.as_tensor(np.diff(np.asarray(row_ptr)), dtype=torch.int64)
    row = torch.repeat_interleave(torch.arange(N), counts)
    col = torch.as_tensor(np.asarray(col), dtype=torch.int64)
    val = torch.as_tensor(np.asarray(val), dtype=F64)
    deg = torch.as_tensor(np.asarray(deg), dtype=F64).reshape(N, 1)
    if norm_max > 0:
        nm = float(norm_max)
    elif norm_max == 0:
        nm = float(set_max_degree)
    else:
        nm = float(deg.max())

    def spmm(rp, c, v, src):
        """sum_j v_ij src[:, j] over the CSR (rp, c, v): [B, N, F] -> [B, N, F]."""
        A = torch.sparse_csr_tensor(rp, c, v, (N, N), check_invariants=False)
        F_ = src.shape[-1]
        return (A @ src.transpose(0, 1).reshape(N, B * F_)).reshape(N, B, F_).transpose(0, 1)

    row_ptr_t = torch.as_tensor(np.asarray(row_ptr), dtype=torch.int64)
    We = W[KEYS[1]]                                        # (63, 8): column 0 multiplies a_ij, 1..7 the x_j
    h = torch.relu(x @ W[KEYS[0]].T)                       # mpnn.py:55
    P = x @ We[:, 1:].T                                    # [B, N, 63]
    # edge stage, mpnn.py:90-100: sum_j ReLU(a_ij w0 + P_j).  Few distinct couplings (integer graphs): one 0/1 product per
    # value a, sum_j [a_ij == a] ReLU(a w0 + P_j); otherwise the edges in chunks.
    values = torch.unique(val)
    emb = torch.zeros(B, N, 63, dtype=F64)
    if len(values) <= 256:
        for a in values:
            m = val == a
            rp = torch.cat([torch.zeros(1, dtype=torch.int64), torch.bincount(row[m], minlength=N).cumsum(0)])
            emb = emb + spmm(rp, col[m], torch.ones(int(m.sum()), dtype=F64), torch.relu(a * We[:, 0] + P))
    else:
        for s in range(0, len(col), chunk):
            r, c, a = row[s:s + chunk], col[s:s + chunk], val[s:s + chunk]
            emb = emb.index_add(1, r, torch.relu(a.view(1, -1, 1) * We[:, 0] + P[:, c]))
    emb = emb / deg
    feat = torch.cat([emb, (deg / nm).expand(B, N, 1)], dim=-1)
    e = torch.relu(feat @ W[KEYS[2]].T)                    # mpnn.py:102
    for layer in range(3):                                 # mpnn.py:68-72, 114-120
        agg = spmm(row_ptr_t, col, val, h) / deg
        msg = torch.relu(torch.cat([agg, e], dim=-1) @ W[KEYS[3 + 2 * layer]].T)
        h = torch.relu(torch.cat([h, msg], dim=-1) @ W[KEYS[4 + 2 * layer]].T)
    pooled = (h.sum(dim=1) / N) @ W[KEYS[9]].T             # mpnn.py:147-157
    f = torch.relu(torch.cat([pooled.unsqueeze(1).expand_as(h), h], dim=-1))
    return (f @ W[KEYS[10]].T + W[KEYS[11]]).squeeze(-1)


def rows_to_x(obs7):
    """Observation rows [B, 7, N] (env.observation(), golden `obs`) -> x [B, N, 7] float64."""
    return torch.as_tensor(np.asarray(obs7), dtype=F64).transpose(1, 2)


def xn_xg_to_x(xn, xg, N):
    """The kernels' inputs xn [B, 3, NP] (rows 0-2) and xg [B, 4] (rows 3-6, one value per episode) -> x [B, N, 7]."""
    xn = torch.as_tensor(np.asarray(xn), dtype=F64)[:, :, :N]
    xg = torch.as_tensor(np.asarray(xg), dtype=F64)
    return torch.cat([xn.transpose(1, 2), xg.unsqueeze(1).expand(-1, N, 4)], dim=-1)
