"""CPU-only checks of the CSR-set Q-network's implementation choice (eco_smpnn_forward_impl, eco_srollout_impl): unknown
impl values, the tensor-core path without packed weights or with a misaligned scratch, and NULL pointers are rejected with
ECO_ERR_INVALID before anything touches a device; engine's host check rejects unpacked weights for TCGEN05."""
import ctypes as C
import types

import pytest

FAKE = C.c_void_p(4096)           # aligned, never dereferenced: every call below fails its argument checks first


@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as ge
    ge.build()
    import eco_dqn_b200
    return eco_dqn_b200.lib()


def weights(_lib, packed):
    w = _lib.Mpnn()
    w.w_init = w.w_edge = w.w_edge_feat = w.w_pool = w.w_read = w.b_read = 4096
    for l in range(3):
        w.w_msg[l] = w.w_upd[l] = 4096
    w.packed = packed
    return w


def bound(L, _lib, n=3000, B=2):
    g, e = _lib.SGraphs(), _lib.Env()
    assert L.eco_sgraphs_bind(C.byref(g), FAKE, 1, n, 10) == 0
    assert L.eco_senv_bind(C.byref(e), FAKE, B, n, 2 * n, -1.0) == 0
    return g, e


def test_forward_impl_rejects_bad_arguments(L):
    import eco_dqn_b200._lib as _lib
    g, _ = bound(L, _lib)

    def fwd(w, impl, xn=FAKE, scratch=FAKE):
        return L.eco_smpnn_forward_impl(C.byref(g), C.byref(w), 2, FAKE, xn, FAKE, 0.0, None, None, scratch, impl, None)

    packed, unpacked = weights(_lib, 4096), weights(_lib, None)
    for impl in (-1, 3, 7):
        assert fwd(packed, impl) == _lib.ECO_ERR_INVALID
        assert b"unknown impl" in L.eco_last_error()
    assert fwd(unpacked, _lib.MPNN_TCGEN05) == _lib.ECO_ERR_INVALID
    assert b"eco_mpnn_pack" in L.eco_last_error()
    assert fwd(packed, _lib.MPNN_TCGEN05, scratch=C.c_void_p(4096 + 16)) == _lib.ECO_ERR_INVALID   # 16- not 32-byte aligned
    assert fwd(packed, _lib.MPNN_TCGEN05, xn=None) == _lib.ECO_ERR_INVALID
    assert b"null" in L.eco_last_error()
    assert L.eco_smpnn_forward_impl(None, C.byref(packed), 2, FAKE, FAKE, FAKE, 0.0, None, None, FAKE, _lib.MPNN_TCGEN05,
                                    None) == _lib.ECO_ERR_INVALID
    w0 = weights(_lib, 4096)
    w0.w_msg[1] = None
    assert fwd(w0, _lib.MPNN_TCGEN05) == _lib.ECO_ERR_INVALID


def test_rollout_impl_rejects_bad_arguments(L):
    import eco_dqn_b200._lib as _lib
    g, e = bound(L, _lib)

    def roll(w, impl, policy=_lib.POLICY_NETWORK, act=FAKE):
        return L.eco_srollout_impl(C.byref(g), C.byref(e), C.byref(w) if w is not None else None, 4, policy, -1.0, act, FAKE,
                                   impl, None, None, None, None)

    packed, unpacked = weights(_lib, 4096), weights(_lib, None)
    assert roll(packed, 5) == _lib.ECO_ERR_INVALID
    assert roll(None, 5, policy=_lib.POLICY_GREEDY) == _lib.ECO_ERR_INVALID       # checked for the greedy policy too
    assert roll(unpacked, _lib.MPNN_TCGEN05) == _lib.ECO_ERR_INVALID
    assert b"eco_mpnn_pack" in L.eco_last_error()
    assert roll(None, _lib.MPNN_TCGEN05) == _lib.ECO_ERR_INVALID
    assert roll(packed, _lib.MPNN_TCGEN05, act=None) == _lib.ECO_ERR_INVALID
    g2, _ = bound(L, _lib, n=2500)
    assert L.eco_srollout_impl(C.byref(g2), C.byref(e), C.byref(packed), 4, _lib.POLICY_NETWORK, -1.0, FAKE, FAKE,
                               _lib.MPNN_TCGEN05, None, None, None, None) == _lib.ECO_ERR_INVALID   # N mismatch


def test_engine_rejects_unpacked_weights_for_tcgen05():
    import eco_dqn_b200._lib as _lib
    import eco_dqn_b200.engine as engine
    env = types.SimpleNamespace(mpnn_impl=_lib.MPNN_AUTO)
    unpacked, packed = types.SimpleNamespace(_packed=None), types.SimpleNamespace(_packed=object())
    with pytest.raises(ValueError):
        engine.BatchedSpinSystem._sparse_impl(env, unpacked, _lib.MPNN_TCGEN05)
    assert engine.BatchedSpinSystem._sparse_impl(env, packed, _lib.MPNN_TCGEN05) == _lib.MPNN_TCGEN05
    assert engine.BatchedSpinSystem._sparse_impl(env, unpacked, None) == _lib.MPNN_AUTO
    assert engine.BatchedSpinSystem._sparse_impl(env, unpacked, _lib.MPNN_SIMT) == _lib.MPNN_SIMT
