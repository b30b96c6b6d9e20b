"""Host canonicalisation of SparseGraphSet's input (engine.sparse_csr) against a dense numpy construction: duplicates resolve
last-writer-wins, edge lists are symmetrised, zeros are dropped, columns are sorted within every row."""
import numpy as np
import pytest
import scipy.sparse as sps

from eco_dqn_b200 import engine


def dense_of(n, row_ptr, col, val, g):
    out = np.zeros((n, n), dtype=np.int64)
    for i in range(n):
        s, e = row_ptr[g * n + i], row_ptr[g * n + i + 1]
        out[i, col[s:e]] = val[s:e]
    return out


def check_canonical(n, row_ptr, col, val):
    assert row_ptr[0] == 0 and row_ptr[-1] == len(col) == len(val)
    assert (np.diff(row_ptr) >= 0).all()
    assert (val != 0).all() and col.dtype == np.int32 and val.dtype == np.int8
    for r in range(len(row_ptr) - 1):
        c = col[row_ptr[r]:row_ptr[r + 1]]
        assert (np.diff(c) > 0).all() and (c >= 0).all() and (c < n).all()


def test_edge_lists_symmetrised_last_writer_wins():
    rng = np.random.default_rng(3)
    n, m = 37, 200
    graphs, want = [], []
    for g in range(3):
        r = rng.integers(0, n, size=m)
        c = rng.integers(0, n, size=m)
        keep = r != c
        r, c = r[keep], c[keep]
        w = rng.integers(-3, 4, size=len(r))             # zeros included: a later zero erases an edge
        A = np.zeros((n, n), dtype=np.int64)
        for i, j, x in zip(r, c, w):                      # the reference's `matrix[i, j] = w; matrix[j, i] = w`, in order
            A[i, j] = x
            A[j, i] = x
        graphs.append((r, c, w))
        want.append(A)
    row_ptr, col, val = engine.sparse_csr(n, graphs)
    check_canonical(n, row_ptr, col, val)
    for g in range(3):
        assert np.array_equal(dense_of(n, row_ptr, col, val, g), want[g])


def test_scipy_and_dense_inputs():
    rng = np.random.default_rng(5)
    n = 50
    A = np.triu(rng.integers(-2, 3, size=(n, n)) * (rng.random((n, n)) < 0.1), 1)
    A = A + A.T
    # a COO matrix with duplicate entries: the last stored one wins (as eco_graphs_load_edges_dev writes them)
    coo = sps.coo_matrix(A)
    r = np.concatenate([coo.row, coo.row[:5]])
    c = np.concatenate([coo.col, coo.col[:5]])
    d = np.concatenate([np.full(len(coo.data), 9), coo.data[:5]])
    d[5:len(coo.data)] = coo.data[5:]
    dup = sps.coo_matrix((d, (r, c)), shape=(n, n))
    for gph in (A, sps.csr_matrix(A), dup):
        row_ptr, col, val = engine.sparse_csr(n, [gph])
        check_canonical(n, row_ptr, col, val)
        assert np.array_equal(dense_of(n, row_ptr, col, val, 0), A)


def test_rejections():
    with pytest.raises(ValueError):
        engine.sparse_csr(32769, [(np.array([0]), np.array([1]), np.array([1]))])
    with pytest.raises(ValueError):
        engine.sparse_csr(0, [])
    with pytest.raises(ValueError):                      # vertex out of range
        engine.sparse_csr(10, [(np.array([0]), np.array([10]), np.array([1]))])
    with pytest.raises(NotImplementedError):             # real-valued couplings
        engine.sparse_csr(10, [(np.array([0]), np.array([1]), np.array([0.5]))])
    with pytest.raises(NotImplementedError):             # outside int8
        engine.sparse_csr(10, [(np.array([0]), np.array([1]), np.array([128]))])


def test_networkx_pickle_entries_without_dense_matrix():
    """load_graph_set_device's N > 2048 route reads a networkx graph through its sparse adjacency: the same entries, in the
    same vertex order, as the dense matrix the reference's loader builds (nx.to_numpy_array)."""
    import networkx as nx
    from eco_dqn_b200.experiments.utils import _sparse_adjacency
    g = nx.gnm_random_graph(60, 200, seed=4)
    rng = np.random.default_rng(4)
    for u, v in g.edges():
        g[u][v]["weight"] = int(rng.choice([-2, -1, 1, 2]))
    g.remove_edge(*next(iter(g.edges())))
    g = nx.relabel_nodes(g, {i: (i * 7) % 60 for i in range(60)})      # node order differs from the labels
    adj = _sparse_adjacency(g)
    assert sps.issparse(adj)
    row_ptr, col, val = engine.sparse_csr(60, [adj])
    assert np.array_equal(dense_of(60, row_ptr, col, val, 0), nx.to_numpy_array(g).astype(np.int64))
