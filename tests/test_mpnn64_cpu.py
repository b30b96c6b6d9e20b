"""Pin the float64 CSR restatement of the Q-network (oracle/mpnn64.py) on the CPU: against the Q the unmodified reference
recorded (tests/golden/*.npz) and against the fp32 row-blocked oracle on +-1, int8 and real-valued graphs.  The GPU
precision tests (test_gpu_q_precision.py) compare every forward kernel and eco_mpnn_grad with this function."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, golden_cases
from oracle.mpnn import KEYS, weights_from_npz, mpnn_forward_blocked
from oracle.mpnn64 import forward64, csr_from_dense, degrees, drop_entry, rows_to_x

# fp32 round-off of the recorded forward.  Observed worst |q64 - q32| / max|q| per episode: 1.9e-6 (golden, er200_g0);
# 7.5e-7 (blocked oracle, 300 vertices, int8 couplings).
PIN_GOLDEN = 4e-6
PIN_BLOCKED = 2e-6


def random_weights(rng, scale=0.3):
    shapes = [(64, 7), (63, 8), (64, 64)] + [(64, 128)] * 6 + [(64, 64), (1, 128), (1,)]
    return {k: (rng.standard_normal(s) * (scale if len(s) > 1 else 0.1)).astype(np.float32) for k, s in zip(KEYS, shapes)}


def per_episode_err(q, ref):
    q, ref = np.asarray(q, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return np.abs(q - ref).max(axis=-1) / np.abs(ref).max(axis=-1)


@pytest.mark.parametrize("name", golden_cases())
def test_forward64_matches_golden_q(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    w = weights_from_npz(z)
    J = z["J"].astype(np.float32)
    csr = csr_from_dense(J)
    deg = degrees(csr[0])
    for si in range(z["obs"].shape[1]):
        q64 = forward64(w, rows_to_x(z["obs"][:, si]), csr, deg, norm_max=-1.0).numpy()
        ref = z["q"][:, si]
        err = per_episode_err(q64, ref)
        assert (err <= PIN_GOLDEN).all(), (name, si, float(err.max()))


@pytest.mark.parametrize("kind", ["pm1", "int8", "real"])
def test_forward64_matches_blocked_oracle(kind):
    rng = np.random.default_rng({"pm1": 1, "int8": 2, "real": 3}[kind])
    n = 300
    up = np.triu(rng.random((n, n)) < 0.1, 1)
    if kind == "pm1":
        vals = np.where(rng.random((n, n)) < 0.5, -1.0, 1.0)
    elif kind == "int8":
        vals = rng.integers(-127, 128, size=(n, n)).astype(np.float64)
    else:
        vals = (2 * rng.random((n, n)) - 1) * 10.0 ** rng.uniform(-6, 3, size=(n, n))
    J = up * vals
    J = (J + J.T).astype(np.float32)
    J[5] = J[:, 5] = 0                                                   # an isolated vertex: degree clamped to 1
    w = random_weights(rng)
    rows = rng.standard_normal((7, n)).astype(np.float32)
    rows[0] = np.sign(rows[0])
    rows[3:] = rows[3:, :1]
    csr = csr_from_dense(J)
    deg = degrees(csr[0])
    for nm in (None, float(deg.max()) + 3.0):
        ref = mpnn_forward_blocked(w, rows.T, J, rows_per_block=64, norm_max=nm).numpy()
        q64 = forward64(w, rows_to_x(rows[None]), csr, deg, norm_max=-1.0 if nm is None else nm).numpy()[0]
        assert per_episode_err(q64, ref) <= PIN_BLOCKED, (kind, nm, float(per_episode_err(q64, ref)))
    # norm_max == 0: the set's maximum degree
    q0 = forward64(w, rows_to_x(rows[None]), csr, deg, norm_max=0.0, set_max_degree=deg.max() + 3.0)
    q3 = forward64(w, rows_to_x(rows[None]), csr, deg, norm_max=deg.max() + 3.0)
    assert torch.equal(q0, q3)


def test_mutants_are_inputs_and_change_q():
    """The three mutants the precision tests assert visible: each is an input, and each moves Q at the vertex it touches."""
    rng = np.random.default_rng(5)
    n, T = 60, 120
    J = np.triu(rng.random((n, n)) < 0.3, 1) * np.where(rng.random((n, n)) < 0.5, -1.0, 1.0)
    J = J + J.T
    w = random_weights(rng)
    x = rows_to_x(np.stack([np.sign(rng.standard_normal((7, n)))] * 2))
    csr = csr_from_dense(J)
    deg = degrees(csr[0])
    hub = int(np.argmax(deg))
    q = forward64(w, x, csr, deg, -1.0)
    dropped = drop_entry(csr, hub)
    assert len(dropped[1]) == len(csr[1]) - 1 and np.array_equal(np.diff(dropped[0])[hub], np.diff(csr[0])[hub] - 1)
    q_drop = forward64(w, x, dropped, deg, -1.0)
    q_dmax = forward64(w, x, csr, deg, float(deg.max()) + 1)
    x_tsf = x.clone()
    x_tsf[:, hub, 2] += 1.0 / T
    q_tsf = forward64(w, x_tsf, csr, deg, -1.0)
    for qm in (q_drop, q_dmax, q_tsf):
        assert (qm[:, hub] - q[:, hub]).abs().min() > 1e-9
    # the dropped entry with the degree recomputed is the graph without that (directed) entry
    Jd = J.copy()
    Jd[hub, csr[1][csr[0][hub + 1] - 1]] = 0
    assert torch.allclose(forward64(w, x, dropped, degrees(dropped[0]), float(deg.max())),
                          forward64(w, x, csr_from_dense(Jd), degrees(csr_from_dense(Jd)[0]), float(deg.max())), rtol=0, atol=1e-12)


def test_forward64_gradients_are_the_directional_derivative():
    """autograd through forward64 (what the eco_mpnn_grad test differentiates) against a central difference of Q."""
    rng = np.random.default_rng(9)
    n = 12
    J = np.triu(rng.random((n, n)) < 0.4, 1) * rng.integers(-3, 4, size=(n, n))
    J = (J + J.T).astype(np.float64)
    csr = csr_from_dense(J)
    deg = degrees(csr[0])
    x = rows_to_x(rng.standard_normal((3, 7, n)))
    w = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in random_weights(rng).items()}
    v = {k: torch.randn_like(t) for k, t in w.items()}
    loss = lambda ww: (forward64(ww, x, csr, deg, -1.0) ** 2).sum()
    loss(w).backward()
    dd = sum(float((w[k].grad * v[k]).sum()) for k in KEYS)
    eps = 1e-6
    with torch.no_grad():
        lp = float(loss({k: w[k] + eps * v[k] for k in KEYS}))
        lm = float(loss({k: w[k] - eps * v[k] for k in KEYS}))
    assert abs((lp - lm) / (2 * eps) - dd) <= 1e-6 * abs(dd)
