"""CSR graph sets (SparseGraphSet) on the device: the gather MPNN forward, the O(degree) env step and [forward + step].

Workloads: synthetic +-1 graphs of the GSet shapes G55 (5000 vertices, 12 498 edges), G70 (10 000 vertices, 9 999 edges) and
G81 (20 000-vertex 2-D torus, 40 000 edges), generated from a seed (the GSet files are not shipped), at B = 128 and B = 1024
episodes, max_steps = 2N.  Per shape and batch: ms per MPNN forward and per env step (CUDA events around every launch of a
profiled rollout of --profile-steps steps), and env-steps/s of an unprofiled rollout of --steps steps.  Then the C4 shape
(2000 vertices, 19 990 +-1 edges, B = 128) through the sparse forward and through the dense tensor-core tile pipeline on the
same graphs (CUDA events around --fwd-calls forwards each), with the largest Q difference between the two.  Prints one JSON
line with the card, its power limit and SM clock read in the same run.

    python tools/bench_sparse.py [--out FILE] [--steps K] [--profile-steps P]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import eco_dqn_b200.engine as engine  # noqa: E402
from eco_dqn_b200 import _lib  # noqa: E402

LINEAR_FLOP_PER_VERTEX = 108530     # 2 * (64*7 + 63*7 + 64*64 + 6 * 64*128 + 128): the per-vertex linears of one forward


def forward_flop(n, nnz, B):
    """linears + gathers (edge stage 3 FLOP per entry and feature, three aggregations 2 per entry and feature)"""
    return B * (LINEAR_FLOP_PER_VERTEX * n + nnz * (63 * 3 + 3 * 64 * 2))


def env_step_bytes(n, deg):
    """csrc/sparse.cu: 6N + 14 d + ~150 bytes per episode-step (ACTIONS policy), d = degree of the flipped vertex"""
    return 6 * n + 14 * deg + 150


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=" + q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, pl, sm, smmax = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit_w": float(pl), "sm_mhz": int(sm), "sm_max_mhz": int(smmax)}
    except Exception as e:     # the card name is still known to the runtime
        return {"name": torch.cuda.get_device_name(), "nvidia_smi": "unavailable (%s)" % e}


def weights(seed=0):
    rng = np.random.default_rng(seed)
    return {k: (rng.standard_normal(s) * (1.0 / np.sqrt(s[-1]))).astype(np.float32)
            for k, s in zip(engine.STATE_DICT_KEYS, engine.STATE_DICT_SHAPES)}


def random_edges(n, m, rng):
    r = rng.integers(0, n, size=3 * m)
    c = rng.integers(0, n, size=3 * m)
    keep = r < c
    pairs = np.unique(np.stack([r[keep], c[keep]], 1), axis=0)
    pairs = pairs[rng.permutation(len(pairs))[:m]]
    return pairs[:, 0], pairs[:, 1], rng.choice(np.array([-1, 1]), size=len(pairs))


def torus(l1, l2, rng):
    idx = np.arange(l1 * l2).reshape(l1, l2)
    r = np.concatenate([idx.ravel(), idx.ravel()])
    c = np.concatenate([np.roll(idx, 1, 0).ravel(), np.roll(idx, 1, 1).ravel()])
    return r, c, rng.choice(np.array([-1, 1]), size=len(r))


def shape(name, rng):
    if name == "G55":
        return 5000, random_edges(5000, 12498, rng)
    if name == "G70":
        return 10000, random_edges(10000, 9999, rng)
    if name == "G81":
        return 20000, torus(100, 200, rng)
    raise ValueError(name)


def run_shape(name, B, w, steps, psteps, L):
    rng = np.random.default_rng({"G55": 55, "G70": 70, "G81": 81}[name])
    n, edges = shape(name, rng)
    gs = engine.SparseGraphSet(n, [edges])
    T = 2 * n
    spins = torch.from_numpy((2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)).cuda()
    env = engine.BatchedSpinSystem(gs, B, T, 1.0 / n)
    out = {"shape": name, "N": n, "edges": gs.nnz // 2, "B": B}
    env.reset(spins=spins)
    env.rollout(w, n_steps=4)                                     # warm-up: module load, every kernel of the timed window
    torch.cuda.synchronize()

    tot, cnt = C.c_double(), C.c_int64()
    env.reset(spins=spins)
    L.eco_profile_enable(1)
    env.rollout(w, n_steps=psteps)
    L.eco_profile_read(0, C.byref(tot), C.byref(cnt))
    out["ms_per_forward"] = tot.value / cnt.value
    L.eco_profile_read(1, C.byref(tot), C.byref(cnt))
    out["ms_per_env_step"] = tot.value / cnt.value
    L.eco_profile_enable(0)
    flop = forward_flop(n, gs.nnz, B)
    out["forward_tflops"] = flop / (out["ms_per_forward"] / 1e3) / 1e12
    out["env_step_bytes_per_episode"] = env_step_bytes(n, gs.nnz / n)
    out["env_step_gbs"] = out["env_step_bytes_per_episode"] * B / (out["ms_per_env_step"] / 1e3) / 1e9

    env.reset(spins=spins)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    env.rollout(w, n_steps=steps)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    out["rollout_steps"] = steps
    out["ms_per_forward_plus_step"] = ms / steps
    out["env_steps_per_s"] = B * steps / (ms / 1e3)
    bc, _, _ = env.results()
    out["mean_best_cut"] = float(bc.float().mean())
    del env, gs
    torch.cuda.empty_cache()
    return out


def time_calls(fn, calls):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


def run_c4(w, calls):
    """C4 shape through both forwards on the same graphs and observations."""
    n, B = 2000, 128
    rng = np.random.default_rng(4)
    r, c, v = random_edges(n, 19990, rng)
    J = np.zeros((n, n), dtype=np.int8)
    J[r, c] = v
    J[c, r] = v
    gd, gsp = engine.GraphSet(J[None]), engine.SparseGraphSet(n, [(r, c, v)])
    spins = (2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)
    ed, es = engine.BatchedSpinSystem(gd, B, 2 * n, 1.0 / n), engine.BatchedSpinSystem(gsp, B, 2 * n, 1.0 / n)
    for e in (ed, es):
        e.reset(spins=spins)
        e.rollout(policy="greedy", n_steps=20)                    # observations away from the all-zero time-since-flip row
    ms_dense = time_calls(lambda: ed.q_values(w), calls)
    ms_sparse = time_calls(lambda: es.q_values(w), calls)
    qd, qs = ed.q_values(w)[0].cpu().numpy(), es.q_values(w)[0].cpu().numpy()
    return {"shape": "C4", "N": n, "edges": gsp.nnz // 2, "B": B, "density": 2 * gsp.nnz / 2 / (n * (n - 1)),
            "ms_per_forward_dense_tc": ms_dense, "ms_per_forward_sparse": ms_sparse, "sparse_over_dense": ms_sparse / ms_dense,
            "max_rel_q_diff": float((np.abs(qs - qd) / np.abs(qd).max(axis=1, keepdims=True)).max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--profile-steps", type=int, default=50)
    ap.add_argument("--fwd-calls", type=int, default=50)
    ap.add_argument("--batches", default="128,1024")
    ap.add_argument("--shapes", default="G55,G70,G81")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sparse.py measures the GPU; no CUDA device found")
    L = _lib.lib()
    res = {"workload": "synthetic +-1 GSet shapes, max_steps = 2N, network policy (gather MPNN, fp32 CUDA cores)",
           "card": card()}
    t0 = time.time()
    w = engine.MPNNWeights(weights())
    res["runs"] = [run_shape(s, int(b), w, args.steps, args.profile_steps, L)
                   for s in args.shapes.split(",") for b in args.batches.split(",")]
    res["c4"] = run_c4(w, args.fwd_calls)
    res["seconds"] = round(time.time() - t0, 1)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
