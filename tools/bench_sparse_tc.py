"""The Q-network of CSR graph sets with its per-vertex linears on the tensor cores (ECO_MPNN_TCGEN05, csrc/sparse_tc.cu) next
to the fp32 gather forward (AUTO), in one process on the same graphs and observations.

Workloads: the synthetic +-1 GSet shapes of tools/bench_sparse.py -- G55 (5000 vertices, 12 498 edges), G70 (10 000, 9 999),
G81 (20 000-vertex torus) -- at B = 128 and 1024, max_steps = 2N, observations of a 20-step Greedy run.  Per shape:
  * ms per forward of each path (CUDA events around --fwd-calls calls, the two paths alternating over --rounds rounds);
  * ms of the seven linears per forward (torch.profiler, a separate window of --prof-calls calls per path);
  * TFLOP/s of the forward, counting 108 530 FLOP per vertex (linears) + 573 per stored entry (gathers);
  * algorithmic GB/s of the linears: 5120 bytes per vertex (K * 4 read + 256 written, seven times);
  * ms per [forward + env step] and env-steps/s of a --steps-step rollout of each path;
  * the largest |q_tc - q_gather| / max|q_gather| of an episode.
Then the C4 shape (2000 vertices, 19 990 edges, B = 128): both sparse forwards next to the dense tile pipeline.  Prints one
JSON line with the card, its power limit and SM clock read in the same run.

    python tools/bench_sparse_tc.py [--out FILE] [--steps K] [--shapes G55,G70,G81] [--batches 128,1024]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import eco_dqn_b200.engine as engine  # noqa: E402
from eco_dqn_b200 import _lib  # noqa: E402
from bench_sparse import LINEAR_FLOP_PER_VERTEX, card, random_edges, shape, weights  # noqa: E402

ENTRY_FLOP = 63 * 3 + 3 * 64 * 2             # 573: edge stage 3 per feature, three aggregations 2 per feature
LINEAR_BYTES_PER_VERTEX = (64 * 4 + 256) + 6 * (128 * 4 + 256)
IMPLS = {"gather": _lib.MPNN_AUTO, "tc": _lib.MPNN_TCGEN05}


def time_fwd(env, w, impl, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        env.q_values(w, impl=impl)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


def linear_ms(env, w, calls):
    """per-forward device time of the linear kernels and of the whole forward's kernels, per path, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for name, impl in IMPLS.items():
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(calls):
                env.q_values(w, impl=impl)
            torch.cuda.synchronize()
        lin = tot = 0.0
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            t = ev.cuda_time_total if t is None else t
            if "k_gemm" in ev.key or "sparse_linear_tc_kernel" in ev.key:
                lin += t
            if any(k in ev.key for k in ("k_gemm", "sparse_linear_tc_kernel", "k_sinit", "k_sgather", "k_sreadout")):
                tot += t
        out[name] = (lin / 1e3 / calls, tot / 1e3 / calls)
    return out


def run_shape(name, B, w, args):
    rng = np.random.default_rng({"G55": 55, "G70": 70, "G81": 81}[name])
    n, edges = shape(name, rng)
    gs = engine.SparseGraphSet(n, [edges])
    T = 2 * n
    spins = torch.from_numpy((2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)).cuda()
    env = engine.BatchedSpinSystem(gs, B, T, 1.0 / n)
    env.reset(spins=spins)
    env.rollout(policy="greedy", n_steps=20)
    out = {"shape": name, "N": n, "edges": gs.nnz // 2, "B": B}
    for impl in IMPLS.values():                                     # warm-up: module load, attributes, scratch
        env.q_values(w, impl=impl)
    torch.cuda.synchronize()
    ms = {k: [] for k in IMPLS}
    for _ in range(args.rounds):
        for k, impl in IMPLS.items():
            ms[k].append(time_fwd(env, w, impl, args.fwd_calls))
    flop = B * (LINEAR_FLOP_PER_VERTEX * n + ENTRY_FLOP * gs.nnz)
    lin = linear_ms(env, w, args.prof_calls)
    for k in IMPLS:
        m = float(np.median(ms[k]))
        out[k] = {"ms_per_forward": m, "ms_per_forward_rounds": ms[k], "forward_tflops": flop / (m / 1e3) / 1e12,
                  "ms_linears_per_forward": lin[k][0], "ms_kernels_per_forward": lin[k][1],
                  "linears_gbs": LINEAR_BYTES_PER_VERTEX * B * n / (lin[k][0] / 1e3) / 1e9,
                  "linears_tflops": LINEAR_FLOP_PER_VERTEX * B * n / (lin[k][0] / 1e3) / 1e12}
    qg, _ = env.q_values(w, impl=IMPLS["gather"])
    qt, _ = env.q_values(w, impl=IMPLS["tc"])
    out["max_rel_q_diff"] = float(((qt - qg).abs().amax(1) / qg.abs().amax(1)).max())
    out["forward_speedup"] = out["gather"]["ms_per_forward"] / out["tc"]["ms_per_forward"]
    for k, impl in IMPLS.items():                                   # [forward + env step]
        env.reset(spins=spins)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        env.rollout(w, n_steps=args.steps, impl=impl)
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1)
        out[k].update({"rollout_steps": args.steps, "ms_per_forward_plus_step": t / args.steps,
                       "env_steps_per_s": B * args.steps / (t / 1e3)})
    del env, gs
    torch.cuda.empty_cache()
    print(json.dumps(out), file=sys.stderr, flush=True)
    return out


def run_c4(w, args):
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
        e.rollout(policy="greedy", n_steps=20)
    runs = {"dense_tc": (ed, _lib.MPNN_AUTO), "sparse_gather": (es, IMPLS["gather"]), "sparse_tc": (es, IMPLS["tc"])}
    for e, impl in runs.values():
        e.q_values(w, impl=impl)
    torch.cuda.synchronize()
    ms = {k: [] for k in runs}
    for _ in range(args.rounds):
        for k, (e, impl) in runs.items():
            ms[k].append(time_fwd(e, w, impl, args.fwd_calls))
    out = {"shape": "C4", "N": n, "edges": gsp.nnz // 2, "B": B}
    out.update({"ms_per_forward_" + k: float(np.median(v)) for k, v in ms.items()})
    out["sparse_tc_over_dense"] = out["ms_per_forward_sparse_tc"] / out["ms_per_forward_dense_tc"]
    qd = ed.q_values(w)[0]
    qs = es.q_values(w, impl=IMPLS["tc"])[0]
    out["max_rel_q_diff_sparse_tc_vs_dense"] = float(((qs - qd).abs().amax(1) / qd.abs().amax(1)).max())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--fwd-calls", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--prof-calls", type=int, default=3)
    ap.add_argument("--batches", default="128,1024")
    ap.add_argument("--shapes", default="G55,G70,G81")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sparse_tc.py measures the GPU; no CUDA device found")
    res = {"workload": "synthetic +-1 GSet shapes, max_steps = 2N; CSR-set Q-network, gather forward (AUTO: fp32 linears) vs "
                       "tensor-core linears (TCGEN05), alternating in one process",
           "card": card()}
    t0 = time.time()
    w = engine.MPNNWeights(weights())
    res["runs"] = [run_shape(s, int(b), w, args) for s in args.shapes.split(",") for b in args.batches.split(",")]
    res["c4"] = run_c4(w, args)
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
