"""The one-launch rollout takes each CTA's episodes through all steps in windows of two (the last window of a CTA with an
odd episode count takes three): it must equal two launches per step (ECO_FUSED_STEP=0) bit for bit, whatever number of
episodes a CTA gets and whether or not the batch is a multiple of the grid.  Every episode has its own graph, so an
operand image or input fetched for the wrong member of a window changes the result."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 200                     # the bench's size: NP = 208, the largest the resident kernel takes

# name -> B as a function of the SM count S (grid = S CTAs; CTA i runs episodes i, i + S, ...)
CASES = {
    "2_per_cta": lambda s: 2 * s,
    "3_per_cta": lambda s: 3 * s,                  # one window of three
    "4_per_cta": lambda s: 4 * s,
    "5_per_cta": lambda s: 5 * s,                  # a window of two, then one of three
    "3_or_2_per_cta": lambda s: 2 * s + 1,         # B not a multiple of the grid: CTA 0 alone has a window of three
    "5_or_4_per_cta": lambda s: 4 * s + s // 2 + 1,
}

_SCRIPT = """
import sys, numpy as np, torch
sys.path.insert(0, %r)
import eco_dqn_b200.engine as eng
from eco_dqn_b200 import _lib
L = _lib.lib()
z = np.load(sys.argv[1])
w = eng.MPNNWeights({k[2:]: z[k] for k in z.files if k.startswith("w_")})
out = {}
for name in z["names"]:
    J, spins = z["J_" + name], z["spins_" + name]
    B, n = spins.shape
    env = eng.BatchedSpinSystem(eng.GraphSet(J), B, 2 * n, 1.0 / n)
    env.reset(spins=spins, graph_idx=np.arange(B, dtype=np.int32))
    torch.cuda.synchronize()
    L.eco_launch_count(1)
    ha, hr, hs = env.rollout(w, record_history=True)
    torch.cuda.synchronize()
    out["launches_" + name] = np.int64(L.eco_launch_count(1))
    bc, bs, st = env.results()
    for k, v in (("best_cut", bc), ("best_spins", bs), ("steps", st), ("ha", ha), ("hr", hr), ("hs", hs), ("xn", env.xn),
                 ("xg", env.xg), ("ep", env._ep)):
        out[k + "_" + name] = v.cpu().numpy()
np.savez(sys.argv[2], **out)
"""


@pytest.fixture(scope="module")
def rollouts(tmp_path_factory):
    """Both paths over every case, each in a child process (ECO_FUSED_STEP is read once per process)."""
    from oracle.mpnn import weights_from_npz
    assert torch.cuda.is_available()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.default_rng(7)
    inputs = {"names": np.array(list(CASES))}
    for name, b_of in CASES.items():
        B = b_of(sms)
        p = rng.uniform(0.05, 0.3, size=(B, 1, 1))                 # degrees (and the per-graph max degree) vary by episode
        upper = np.triu(rng.random((B, N, N)) < p, 1)
        sign = np.where(rng.random((B, N, N)) < 0.5, -1, 1)
        J = (upper * sign).astype(np.int8)
        inputs["J_" + name] = J + J.transpose(0, 2, 1)
        inputs["spins_" + name] = (2 * rng.integers(0, 2, size=(B, N)) - 1).astype(np.int8)
    wd = weights_from_npz(np.load(os.path.join(ROOT, "tests", "golden", "er200_g0.npz")))
    inputs.update({"w_" + k: v for k, v in wd.items()})
    tmp = tmp_path_factory.mktemp("rollout_window")
    inp = str(tmp / "in.npz")
    np.savez(inp, **inputs)
    res = {}
    for tag, flag in (("two", "0"), ("fused", "1")):
        out = str(tmp / (tag + ".npz"))
        subprocess.run([sys.executable, "-c", _SCRIPT % ROOT, inp, out], check=True,
                       env=dict(os.environ, ECO_FUSED_STEP=flag), timeout=600)
        res[tag] = dict(np.load(out))
    return res


@pytest.mark.parametrize("case", list(CASES))
def test_windowed_one_launch_rollout_equals_two_launches_per_step(rollouts, case):
    two, fused = rollouts["two"], rollouts["fused"]
    steps = 2 * N
    assert fused["launches_" + case] == 1, "the rollout did not run as one launch"
    assert two["launches_" + case] >= 2 * steps
    for k in ("best_cut", "best_spins", "steps", "ha", "hr", "hs", "xn", "xg", "ep"):
        a, b = two[k + "_" + case], fused[k + "_" + case]
        assert a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)), k
    assert (two["steps_" + case] == steps).all() and (two["ha_" + case] >= 0).all()
