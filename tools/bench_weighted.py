"""Real-valued couplings (EdgeType.RANDOM) on the device: the weighted rollout and the fp64 env-step kernel alone.

Workload: ER-200 (p = 0.15) with 2*rand-1 weights, G = 4096 distinct graphs (1.3 GB of fp64 couplings, larger than L2),
B = 4096 episodes (episode b on graph b), T = 400 steps of the network policy.  Prints one JSON line with the card, its power
limit and SM clock (read in the same run), ms per MPNN forward and per env step (CUDA events around every launch of a
separate profiled rollout), env-steps/s of an unprofiled rollout, and the env kernel alone at B = 262 144 as algorithmic
bytes/s (39.25 N + 96 per episode-step, csrc/weighted.cu) over the 6533.5 GB/s HBM copy peak of DESIGN.md section 4.1.

    python tools/bench_weighted.py [--out FILE]
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

HBM_COPY_GBS = 6533.5       # DESIGN.md section 4.1: measured device-to-device copy rate of the B200


def bytes_env_weighted(n):
    """Algorithmic bytes of one weighted episode-step: row a of fp64 J, spins, fp64 fields read + write, last-flip steps,
    best-diff bits, three fp32 feature rows, scalar block."""
    return 8 * n + n + 16 * n + 2 * n + 2 * ((n + 7) // 8) + 12 * n + 96


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=" + q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, pl, sm, smmax = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit_w": float(pl), "sm_mhz": int(sm), "sm_max_mhz": int(smmax)}
    except Exception as e:     # the card name is still known to the runtime
        return {"name": torch.cuda.get_device_name(), "nvidia_smi": "unavailable (%s)" % e}


def random_er(count, n, p, seed):
    from eco_dqn_b200.envs.utils import EdgeType, RandomErdosRenyiGraphGenerator
    import random
    random.seed(seed)
    np.random.seed(seed)
    gen = RandomErdosRenyiGraphGenerator(n, p, EdgeType.RANDOM)
    return np.stack([gen.get() for _ in range(count)])


def weights(seed=0):
    rng = np.random.default_rng(seed)
    return {k: (rng.standard_normal(s) * (1.0 / np.sqrt(s[-1]))).astype(np.float32)
            for k, s in zip(engine.STATE_DICT_KEYS, engine.STATE_DICT_SHAPES)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--graphs", type=int, default=4096)
    ap.add_argument("--episodes", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--env-episodes", type=int, default=262144)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_weighted.py measures the GPU; no CUDA device found")
    n, G, B, T = 200, args.graphs, args.episodes, args.steps
    L = _lib.lib()
    res = {"workload": "ER-200 p=0.15 EdgeType.RANDOM, G=%d, B=%d, T=%d, network policy (SIMT MPNN on fp32 J)" % (G, B, T),
           "card": card()}

    t0 = time.time()
    Js = random_er(G, n, 0.15, seed=0)
    gs = engine.WeightedGraphSet(Js)
    del Js
    res["graph_set_gb"] = round(gs._ws.numel() / 1e9, 3)
    w = engine.MPNNWeights(weights(), pack=False)
    rng = np.random.default_rng(1)
    spins = torch.from_numpy((2 * rng.integers(0, 2, size=(B, n)) - 1).astype(np.int8)).cuda()
    gidx = torch.arange(B, dtype=torch.int32, device="cuda") % G
    env = engine.BatchedSpinSystem(gs, B, T, 1.0 / n)
    res["setup_s"] = round(time.time() - t0, 1)

    # warm-up (module load, every kernel of the timed window)
    env.reset(spins=spins, graph_idx=gidx)
    env.rollout(w, n_steps=4)
    torch.cuda.synchronize()

    # per-kernel device time: every forward and env-step launch bracketed by events
    env.reset(spins=spins, graph_idx=gidx)
    L.eco_profile_enable(1)
    env.rollout(w, n_steps=T)
    tot, cnt = C.c_double(), C.c_int64()
    L.eco_profile_read(0, C.byref(tot), C.byref(cnt))            # kind 0: MPNN forward
    res["ms_per_forward"] = tot.value / cnt.value
    L.eco_profile_read(1, C.byref(tot), C.byref(cnt))                          # kind 1: env step
    res["ms_per_env_step"] = tot.value / cnt.value
    L.eco_profile_enable(0)

    # end to end, profiler off
    env.reset(spins=spins, graph_idx=gidx)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    env.rollout(w, n_steps=T)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    res["rollout_ms"] = ms
    res["env_steps_per_s"] = B * T / (ms / 1e3)
    bc, _, _ = env.results()
    res["mean_best_cut"] = float(bc.mean())
    del env

    # env kernel alone, HBM-bound size (random actions, caller-supplied)
    BE = args.env_episodes
    enva = engine.BatchedSpinSystem(gs, BE, T, 1.0 / n)
    sp = torch.from_numpy((2 * rng.integers(0, 2, size=(BE, n)) - 1).astype(np.int8)).cuda()
    enva.reset(spins=sp, graph_idx=torch.arange(BE, dtype=torch.int32, device="cuda") % G)
    gen = torch.Generator(device="cuda").manual_seed(7)
    acts = [torch.randint(0, n, (BE,), generator=gen, device="cuda", dtype=torch.int32) for _ in range(44)]
    for a in acts[:4]:
        enva.step(a)
    torch.cuda.synchronize()
    L.eco_profile_enable(1)
    for a in acts[4:]:
        enva.step(a)
    L.eco_profile_read(1, C.byref(tot), C.byref(cnt))
    L.eco_profile_enable(0)
    s = tot.value / cnt.value / 1e3
    gbs = bytes_env_weighted(n) * BE / s / 1e9
    res["env_kernel"] = {"B": BE, "us_per_launch": s * 1e6, "env_steps_per_s": BE / s, "bytes_per_step": bytes_env_weighted(n),
                         "algorithmic_gbs": gbs, "frac_of_hbm_copy_peak": gbs / HBM_COPY_GBS}
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
