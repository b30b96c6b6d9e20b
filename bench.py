#!/usr/bin/env python
"""bench.py -- env-steps/sec incl. MPNN Q-eval for the batched ECO-DQN Max-Cut rollout (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, one process per GPU)
    python bench.py --impl reference --steps K --warmup W    # reference arm: the reference's own CPU code on host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as DIR/*.npy

One bench "step" = one full greedy-Q rollout of a batch: reset + T = 2N env steps for B episodes, each env step being one
MPNN Q-evaluation + argmax + one fused env-step kernel.  Headline workload = the configuration BASELINE.json's `metric` is
quoted on: ER-200 (G(200, 0.15), +-1 weights), B = 4096 concurrent episodes per GPU, 4096 distinct graphs per GPU (int8
adjacency 164 MB + bf16 operand images 708 MB > the 126 MB L2, so no L2 flush is needed between iterations), the
reference's pretrained ER_200spin checkpoint, every episode normalised by its own graph like the reference's per-graph
batches.  The other BASELINE configs ride on the same line as side blocks measured on rank 0: `c2_ba200` (configs[1]: same
size, Barabasi-Albert graphs -- the kernels are density-independent), `c1_er20`, `c3_er500`, `c4_gset2000`, `c5_dqn`; with
--gpus N > 1 every rank also runs C3 sharded (4096 ER-500 episodes per GPU, best cuts all-gathered) and the C5
data-parallel DQN.learn (one gradient all-reduce per update).  Prints ONE JSON line on rank 0.
"""
import argparse
import contextlib
import io
import json
import os
import random
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env-steps/sec incl. MPNN Q-eval"
N_SPINS = 200
ER_P = 0.15
BA_M = 4
B_PER_GPU = 4096
CPU_SAMPLE = (16, 0.5)     # reference arm / cpu_baseline: episodes of ONE graph, step_factor (T = 100 env steps each)
PROFILE_STRIDE = 8         # kernel launches bracketed by CUDA events inside the timed region: one in 8


def flops_mpnn(n):
    """SURVEY.md section 8(d): algorithmic flops of one Q-evaluation of one episode (+-1 graphs)."""
    return 636 * n * n + 108530 * n + 8192


def bytes_env(n):
    """SURVEY.md section 8(d): algorithmic bytes of one env step of one episode (features materialised)."""
    return 20.25 * n + 96


# ---------------------------------------------------------------------------------------------------------------------
# synthetic graphs (the reference's generators, src/envs/utils.py:165-236, EdgeType.DISCRETE)
# ---------------------------------------------------------------------------------------------------------------------
def ba_graphs(count, n, m, seed):
    """BA(n, m) graphs with +-1 weights, like RandomBarabasiAlbertGraphGenerator (reference src/envs/utils.py:204-236)."""
    import networkx as nx
    np.random.seed(seed)
    random.seed(seed)
    out = np.zeros((count, n, n), dtype=np.int8)
    for i in range(count):
        g = nx.barabasi_albert_graph(n, m)
        adj = nx.to_numpy_array(g)
        mask = 2. * np.random.randint(2, size=(n, n)) - 1.
        mask = np.tril(mask) + np.triu(mask.T, 1)
        a = adj * mask
        np.fill_diagonal(a, 0)
        out[i] = a.astype(np.int8)
    return out


def er_graphs(count, n, p, seed):
    """G(n, p) graphs with +-1 weights, like RandomErdosRenyiGraphGenerator with EdgeType.DISCRETE (reference
    src/envs/utils.py:165-202: a symmetric Bernoulli(p) mask times a symmetric +-1 matrix, zero diagonal)."""
    rng = np.random.default_rng(seed)
    out = np.zeros((count, n, n), dtype=np.int8)
    iu = np.triu_indices(n, 1)
    for i in range(count):
        keep = rng.random(len(iu[0])) < p
        sign = (2 * rng.integers(0, 2, size=len(iu[0])) - 1).astype(np.int8)
        out[i, iu[0], iu[1]] = keep * sign
        out[i] += out[i].T
    return out


def gnm_graphs(count, n, edges, seed):
    """GSet-shaped instances (G22-G31: 2000 vertices, 19 990 edges, +-1 weights): `edges` random vertex pairs, random signs.
    The shipped gset pickles are missing from the reference tree (.MISSING_LARGE_BLOBS), so synthetic only."""
    rng = np.random.default_rng(seed)
    out = np.zeros((count, n, n), dtype=np.int8)
    iu = np.triu_indices(n, 1)
    for i in range(count):
        pick = rng.choice(len(iu[0]), size=edges, replace=False)
        out[i, iu[0][pick], iu[1][pick]] = (2 * rng.integers(0, 2, size=edges) - 1).astype(np.int8)
        out[i] += out[i].T
    return out


def load_weights(name="ba200_g0"):
    """A pretrained reference checkpoint as recorded in a golden fixture (`w::<key>`): ba200_g0 -> eco/network_best_BA_200spin,
    er200_g0 -> ER_200spin, er20_g0 -> ER_20spin."""
    z = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    return {k[3:]: np.asarray(z[k], dtype=np.float32) for k in z.files if k.startswith("w::")}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d["bf16_tflops_sustained"], "tflops_burst": d["bf16_tflops"],
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "tflops_burst": 1590.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU baseline: the reference itself (oracle/_ref, vendored by oracle/make_ref.py) or, without it, the oracle port
# ---------------------------------------------------------------------------------------------------------------------
def eco_env_args(mod, n):
    return {'observables': mod.DEFAULT_OBSERVABLES, 'reward_signal': mod.RewardSignal.BLS,
            'extra_action': mod.ExtraAction.NONE, 'optimisation_target': mod.OptimisationTarget.CUT,
            'spin_basis': mod.SpinBasis.SIGNED, 'norm_rewards': True, 'memory_length': None, 'horizon_length': None,
            'stag_punishment': None, 'basin_reward': 1. / n, 'reversible_spins': True, 'stopping': mod.Stopping.NORMAL}


class CpuReference:
    """The reference's CPU path on a bounded sample: `n_eps` episodes of ONE graph (the reference batches the attempts of
    one graph), T = step_factor * N env steps each, torch CPU threads = all host cores.  kind "reference": the unmodified
    reference's test_network (experiments/utils.py:22-303) from oracle/_ref -- the value is T / its own `time` column, i.e.
    its own timer around the network rollout loop (reset, greedy baselines and numba warm-up excluded, :164,214).  kind
    "port": oracle.rollout, when oracle/_ref is absent."""

    def __init__(self):
        import torch
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        self.kind, self.why_port = "port", "oracle/_ref absent"
        try:
            from oracle import make_ref
            if make_ref.import_reference():
                import src.envs.utils as ref_utils
                from src.networks.mpnn import MPNN
                from experiments.utils import test_network
                self.ref_utils, self.MPNN, self.test_network = ref_utils, MPNN, test_network
                self.kind = "reference"
        except Exception as e:          # e.g. numba missing on some box: fall back to the port and say so
            self.why_port = "%s: %s" % (type(e).__name__, e)

    def network(self, weights):
        import torch
        net = self.MPNN(n_obs_in=7, n_layers=3, n_features=64, n_hid_readout=[], tied_weights=False)
        net.load_state_dict({k: torch.tensor(v) for k, v in weights.items()})
        net.eval()
        for p in net.parameters():
            p.requires_grad = False
        return net

    def run(self, J, weights, n_eps, step_factor, seed=0):
        """-> (env-steps/s of the rollout loop, seconds of that loop)."""
        n = J.shape[0]
        T = int(n * step_factor)
        if self.kind == "reference":
            np.random.seed(seed)
            with contextlib.redirect_stdout(io.StringIO()):
                res = self.test_network(self.network(weights), eco_env_args(self.ref_utils, n), [J.astype(np.float64)], "cpu",
                                        step_factor, n_attempts=n_eps)
            per_attempt = float(res["time"][0])          # t_total / n_attempts (experiments/utils.py:270)
            return T / per_attempt, per_attempt * n_eps
        from oracle.rollout import rollout as cpu_rollout
        rng = np.random.default_rng(seed)
        spins = (2 * rng.integers(0, 2, size=(n_eps, n)) - 1).astype(np.int8)
        out = cpu_rollout(J.astype(np.float64), weights, spins, T, 1.0 / n)
        return out["env_steps"] / out["seconds"], out["seconds"]

    def warm(self, J, weights):
        self.run(J, weights, 2, 4.0 / J.shape[0])           # numba JIT, thread pools, allocator

    def describe(self, n_eps, step_factor, n, secs=None):
        s = "%d episodes x %d env steps of one ER-%d graph per bench step, batched like the reference's test_network" % (
            n_eps, int(n * step_factor), n)
        if secs is not None:
            s += " (%.1f s of CPU work)" % secs
        return s


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = N_SPINS
    weights = load_weights("er200_g0")
    J = er_graphs(1, n, ER_P, seed=0)[0]
    n_eps, sf = CPU_SAMPLE
    cpu = CpuReference()
    cpu.warm(J, weights)
    for i in range(args.warmup):
        cpu.run(J, weights, 2, 8.0 / n, seed=i)
    vals = []
    t0 = time.perf_counter()
    for i in range(args.steps):
        v, _ = cpu.run(J, weights, n_eps, sf, seed=100 + i)
        vals.append(v)
    wall = time.perf_counter() - t0
    value = float(np.mean(vals))
    sample = cpu.describe(n_eps, sf, n)
    config = {"workload": "ER_200spin (p=0.15, +-1 weights) ECO-DQN greedy-Q rollout on the host CPU: BOUNDED SAMPLE of the "
                          "product arm's workload -- " + sample + "; the full step (4096 episodes x 400 steps) is infeasible "
                          "on the CPU",
              "step": "one call of the reference's test_network on one graph: value = T / its `time` column (its own timer "
                      "around the network rollout loop)",
              "n_spins": n, "episodes_per_step": n_eps, "env_steps_per_episode": int(n * sf),
              "weights": "pretrained eco/network_best_ER_200spin (reference checkpoint)",
              "implementation": "unmodified reference from oracle/_ref (oracle/make_ref.py)" if cpu.kind == "reference"
                                else "oracle port (%s)" % cpu.why_port}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * wall / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cpu.cores, "kind": cpu.kind, "sample": sample},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
# C5: DQN training
# ---------------------------------------------------------------------------------------------------------------------
def dqn_update_sample(timesteps=3000, n_envs=16):
    """C5 of BASELINE.json: DQN.learn on ER-40 with the hyper-parameters of experiments/train_eco.py (minibatch 64 per rank,
    update every 32 steps, replay 5000).  Returns ms per train_step (TD target + eco_mpnn_grad [+ all-reduce] + Adam) and ms
    per 1000 environment timesteps of the whole learn loop, per rank.  With several ranks every update carries ONE gradient
    all-reduce; the parameters of all ranks must stay bit-identical.  A reported side number, not the bench metric."""
    import tempfile
    import torch
    import torch.distributed as dist
    import eco_dqn_b200.envs.core as ising_env
    from eco_dqn_b200.envs.utils import (DEFAULT_OBSERVABLES, RewardSignal, ExtraAction, OptimisationTarget, SpinBasis,
                                         Stopping, RandomErdosRenyiGraphGenerator, EdgeType)
    from eco_dqn_b200.networks.mpnn import MPNN
    from eco_dqn_b200.agents.dqn.dqn import DQN
    from eco_dqn_b200.agents.dqn.utils import TestMetric
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    n = 40
    env_args = {'observables': DEFAULT_OBSERVABLES, 'reward_signal': RewardSignal.BLS, 'extra_action': ExtraAction.NONE,
                'optimisation_target': OptimisationTarget.CUT, 'spin_basis': SpinBasis.SIGNED, 'norm_rewards': True,
                'memory_length': None, 'horizon_length': None, 'stag_punishment': None, 'basin_reward': 1. / n,
                'reversible_spins': True, 'stopping': Stopping.NORMAL}
    with contextlib.redirect_stdout(sys.stderr):
        env = ising_env.make("SpinSystem", RandomErdosRenyiGraphGenerator(n, 0.15, EdgeType.DISCRETE), 2 * n, **env_args)
        tmp = tempfile.mkdtemp()
        agent = DQN([env], lambda: MPNN(), init_weight_std=0.01, double_dqn=True, gamma=0.95, update_learning_rate=False,
                    initial_learning_rate=1e-4, minibatch_size=64, update_frequency=32, update_target_frequency=1000,
                    replay_start_size=500, replay_buffer_size=5000, final_exploration_step=3000,
                    final_exploration_rate=0.05, test_frequency=10 ** 9, save_network_frequency=10 ** 9, logging=False,
                    seed=5, test_metric=TestMetric.BEST, test_save_path=os.path.join(tmp, "s%d" % rank),
                    network_save_path=os.path.join(tmp, "n%d" % rank), n_envs=n_envs)
        acc = {"s": 0.0, "n": 0}
        orig = agent._train_step_device      # what learn() calls: the update for a set of replay rows, loss kept on the device

        def timed(tr):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = orig(tr)
            torch.cuda.synchronize()
            acc["s"] += time.perf_counter() - t0
            acc["n"] += 1
            return out

        agent._train_step_device = timed
        agent.learn(timesteps=1000)          # warm-up: fills the replay, first updates (captures the update's CUDA graph)
        acc["s"], acc["n"] = 0.0, 0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        agent.learn(timesteps=timesteps)
        torch.cuda.synchronize()
        tot = time.perf_counter() - t0
    out = {"workload": "DQN.learn, ER-40 p=0.15, minibatch 64 per rank, update every 32 timesteps, %d lock-step environments "
                       "per rank" % n_envs,
           "ranks": world, "train_step_ms": acc["s"] / max(acc["n"], 1) * 1e3, "train_steps": acc["n"],
           "ms_per_1000_timesteps": tot / timesteps * 1e6, "timing": "host clock around synchronised calls"}
    if world > 1:
        flat = torch.cat([p.detach().reshape(-1) for p in agent.network.parameters()])
        gathered = [torch.zeros_like(flat) for _ in range(world)]
        dist.all_gather(gathered, flat)
        out["params_identical_across_ranks"] = bool(all(torch.equal(gathered[0], g) for g in gathered))
        # the collective alone: the flat 58 425-float gradient buffer, like sharding.allreduce_mean_
        buf = torch.zeros(flat.numel(), dtype=torch.float32, device=flat.device)
        for _ in range(10):
            dist.all_reduce(buf)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(100):
            dist.all_reduce(buf)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) * 10.0], dtype=torch.float64, device=flat.device)       # us per all-reduce
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out["allreduce_us"] = float(t.item())
        out["allreduce_bytes"] = int(flat.numel() * 4)
        ts = torch.tensor([out["train_step_ms"], out["ms_per_1000_timesteps"]], dtype=torch.float64, device=flat.device)
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        out["train_step_ms"], out["ms_per_1000_timesteps"] = float(ts[0].item()), float(ts[1].item())
    return out


# ---------------------------------------------------------------------------------------------------------------------
# product arm
# ---------------------------------------------------------------------------------------------------------------------
def headline_config(world):
    return {"workload": "ER_200spin (G(200, 0.15), +-1 weights) batched ECO-DQN greedy-Q rollout, %d concurrent episodes per GPU, "
                        "%d distinct graphs per GPU, T=2N=%d env steps per episode; BASELINE configs[1] (BA_200spin, same size) "
                        "is the side block c2_ba200" % (B_PER_GPU, B_PER_GPU, 2 * N_SPINS),
            "step": "one full rollout: reset + T x (MPNN Q-eval + argmax + env step) for the whole batch",
            "n_spins": N_SPINS, "episodes_per_gpu": B_PER_GPU, "env_steps_per_episode": 2 * N_SPINS,
            "graphs_per_gpu": B_PER_GPU, "weights": "pretrained eco/network_best_ER_200spin (reference checkpoint)",
            "normalisation": "per graph (mpnn.py:102 over the reference's one-graph batches)",
            "l2": "inputs larger than L2 (per GPU: bf16 adjacency operand images 708 MB + int8 adjacency 177 MB + 50 MB state); no flush needed",
            "parallelism": "episodes sharded over %d GPU(s), no collective during rollout, all_gather of best cuts" % world}


def dump_outputs(out_dir, arrays):
    """out_dir/<name>.npy for each device tensor of `arrays`, as float64 (exact for the int32 / int8 results), so that
    the outputs of two builds can be compared array for array."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist
    import eco_dqn_b200.engine as engine
    from eco_dqn_b200 import _lib
    import ctypes as C

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = _lib.lib()
    impl = {"auto": _lib.MPNN_AUTO, "simt": _lib.MPNN_SIMT, "tc": _lib.MPNN_TCGEN05}[args.mpnn]
    pk = peaks()
    tot, cnt = C.c_double(), C.c_int64()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def prof_read(kind):
        L.eco_profile_read(kind, C.byref(tot), C.byref(cnt))
        return tot.value, cnt.value

    class Rollout:
        """One workload: graphs + B episodes + weights; step() = reset + full rollout (+ the best-cut gather)."""

        def __init__(self, J, B, T, wd, seed, gather=True):
            self.n, self.B, self.T = J.shape[1], B, T
            self.gs = engine.GraphSet(J)
            self.env = engine.BatchedSpinSystem(self.gs, B, T, 1.0 / self.n, mpnn_impl=impl)
            self.w = engine.MPNNWeights(wd)
            rng = np.random.default_rng(seed)
            self.spins = torch.from_numpy((2 * rng.integers(0, 2, size=(B, self.n)) - 1).astype(np.int8)).cuda()
            self.gidx = (torch.arange(B, dtype=torch.int32, device="cuda") % J.shape[0]).contiguous()
            self.gathered = [torch.empty(B, dtype=torch.int32, device="cuda") for _ in range(world)] \
                if (world > 1 and gather) else None
            self.used_impl = "tcgen05" if (impl != _lib.MPNN_SIMT and self.w.c.packed and self.gs.pm1_only) else "simt"

        def step(self, n_steps=None):
            """-> results() of the rollout: best cut [B], best spins [B, n], steps taken [B]."""
            self.env.reset(spins=self.spins, graph_idx=self.gidx)
            self.env.rollout(self.w, n_steps=n_steps)
            res = self.env.results()
            if self.gathered is not None:
                dist.all_gather(self.gathered, res[0])         # the path's only collective: final best cuts
            return res

        def timed(self, warmup, steps, n_steps=None, sample_clocks=False):
            """-> dict(ms_total over `steps` rollouts (max over ranks), mpnn / env kernel averages, launches)."""
            for _ in range(warmup):
                self.step(n_steps)
            barrier()
            L.eco_launch_count(1)
            L.eco_profile_enable(PROFILE_STRIDE)
            sampler = ClockSampler(local) if sample_clocks else None
            if sampler:
                sampler.start()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            ev0.record()
            for _ in range(steps):
                res = self.step(n_steps)
            ev1.record()
            barrier()
            clocks = sampler.stop() if sampler else None
            ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            launches = int(L.eco_launch_count(0))
            mpnn_ms, mpnn_n = prof_read(0)
            env_ms, env_n = prof_read(1)
            roll_ms, roll_n = prof_read(2)      # one-launch rollouts: total time, rollout STEPS covered
            L.eco_profile_enable(0)
            one_launch = roll_n > 0
            if one_launch:                      # per step: forward + argmax + env step inside the resident kernel
                mpnn_ms, mpnn_n, env_ms, env_n = roll_ms, roll_n, 0.0, 0
            return {"ms_total": float(ms.item()), "mpnn_ms": mpnn_ms / max(mpnn_n, 1), "mpnn_n": mpnn_n,
                    "env_ms": env_ms / max(env_n, 1), "env_n": env_n, "launches": launches, "clocks": clocks, "best": res[0],
                    "results": res, "one_launch": one_launch}

        def side_block(self, name, r, steps, env_steps_per_rollout, ranks=1):
            """ms per [MPNN + env step], env-steps/s, roofline fraction of the MPNN forward of this size."""
            ach = flops_mpnn(self.n) * self.B / (r["mpnn_ms"] / 1e3) / 1e12
            return {"workload": name, "n_spins": self.n, "episodes_per_gpu": self.B, "env_steps_per_episode": self.T,
                    "graphs_per_gpu": self.gs.G, "gpus": ranks, "mpnn_impl": self.used_impl,
                    "env_steps_per_s": ranks * env_steps_per_rollout * steps / (r["ms_total"] / 1e3),
                    "ms_per_env_step_launch_pair": r["ms_total"] / steps / (env_steps_per_rollout / self.B),
                    "mpnn_forward_ms": r["mpnn_ms"], "env_step_us": None if r["one_launch"] else r["env_ms"] * 1e3,
                    "launches_per_rollout": "1 (forward + argmax + env step of all steps in one kernel)" if r["one_launch"]
                    else "2 per step",
                    "roofline": {"bound": "tensor", "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s",
                                 "frac": ach / pk["tflops"], "flops_per_launch": flops_mpnn(self.n) * self.B},
                    "mean_best_cut": float(r["best"].float().mean().item())}

    # ---- headline: ER-200 -------------------------------------------------------------------------------------------
    n, T, B, G = N_SPINS, 2 * N_SPINS, B_PER_GPU, B_PER_GPU
    wd = load_weights("er200_g0")
    J = er_graphs(G, n, ER_P, seed=rank)                      # each rank owns its own graphs + episodes
    head = Rollout(J, B, T, wd, seed=1000 + rank)
    r = head.timed(args.warmup, args.steps, sample_clocks=True)
    ms_total, bc = r["ms_total"], r["best"]
    value = world * B * T * args.steps / (ms_total / 1000.0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("best_cut", "best_spins", "steps"), r["results"])))

    # ---- the env-step kernel alone at the bench's batch (the rollout applies the step inside the MPNN kernel) ----
    env_small = None
    if rank == 0:
        gen = torch.Generator(device="cuda").manual_seed(11)
        acts = [torch.randint(0, n, (B,), generator=gen, device="cuda", dtype=torch.int32) for _ in range(36)]
        head.env.reset(spins=head.spins, graph_idx=head.gidx)
        for a in acts[:4]:
            head.env.step(a)
        torch.cuda.synchronize()
        L.eco_profile_enable(1)
        for a in acts[4:]:
            head.env.step(a)
        ems, en = prof_read(1)
        L.eco_profile_enable(0)
        env_small = (ems / max(en, 1), en)

    # ---- e2e: host buffers in, host buffers out, through the C-ABI session (H2D + D2H inside the timing) ----
    sess = engine.HostSession(G, n, B, T, 1.0 / n, wd, impl=impl)
    J_pin = torch.from_numpy(J).pin_memory()
    spins_pin = head.spins.cpu().pin_memory()
    gidx_pin = head.gidx.cpu().pin_memory()
    cut_pin = torch.zeros(B, dtype=torch.int32).pin_memory()
    bs_pin = torch.zeros(B, n, dtype=torch.int8).pin_memory()
    e2e_steps = max(1, min(args.steps, 3))
    sess.rollout(J_pin, gidx_pin, spins_pin, cut_pin, bs_pin)          # warm-up
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        sess.rollout(J_pin, gidx_pin, spins_pin, cut_pin, bs_pin)
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * B * T * e2e_steps / float(e2e_s.item())
    assert np.array_equal(cut_pin.numpy(), bc.cpu().numpy()), "session result differs from engine result"
    sess.close()

    # ---- env-step kernel alone at a size that is HBM- rather than launch-bound ---------------------------
    env_only = None
    if rank == 0 and not args.skip_env_only and world == 1:
        Bbig = 262144
        rng = np.random.default_rng(5)
        envb = engine.BatchedSpinSystem(head.gs, Bbig, T, 1.0 / n)
        envb.reset(spins=torch.from_numpy((2 * rng.integers(0, 2, size=(Bbig, n)) - 1).astype(np.int8)).cuda())
        gen = torch.Generator(device="cuda").manual_seed(7)
        acts = [torch.randint(0, n, (Bbig,), generator=gen, device="cuda", dtype=torch.int32) for _ in range(24)]
        for a in acts[:4]:
            envb.step(a)
        torch.cuda.synchronize()
        L.eco_profile_enable(1)
        for a in acts[4:]:
            envb.step(a)
        ems, en = prof_read(1)
        L.eco_profile_enable(0)
        avg = ems / en / 1000.0
        gbs = bytes_env(n) * Bbig / avg / 1e9
        env_only = {"episodes": Bbig, "avg_launch_us": avg * 1e6, "env_steps_per_s": Bbig / avg,
                    "achieved_gbs": gbs, "peak_gbs": pk["hbm_gbs"], "frac": gbs / pk["hbm_gbs"],
                    "bytes_per_env_step": bytes_env(n)}
        del envb

    # ---- the other BASELINE configs ----------------------------------------------------------------------------------
    side = {}
    if not args.skip_sizes:
        try:
            if world == 1:
                c2 = Rollout(ba_graphs(256, n, BA_M, seed=0), B, T, load_weights("ba200_g0"), seed=2)
                side["c2_ba200"] = c2.side_block("BA_200spin (m=4, +-1), configs[1]: 4096 episodes over 256 distinct graphs",
                                                 c2.timed(1, 2), 2, B * T)
                del c2
                n1 = 20
                c1 = Rollout(er_graphs(100, n1, 0.15, seed=0), 5000, 2 * n1, load_weights("er20_g0"), seed=3)
                side["c1_er20"] = c1.side_block("ER_20spin greedy test rollout, configs[0]: 100 graphs x 50 random inits, 2N steps "
                                                "(tcgen05 kernel packs 6 graphs per CTA pass)", c1.timed(2, 5), 5, 5000 * 2 * n1)
                del c1
                n4 = 2000
                c4 = Rollout(gnm_graphs(8, n4, 19990, seed=0), 128, 2 * n4, wd, seed=4)
                side["c4_gset2000"] = c4.side_block("GSet-shaped 2000-vertex +-1 graphs (19 990 edges), configs[3]: 128 episodes over "
                                                    "8 graphs, 2N = 4000 steps (dense operand-tile pipeline)",
                                                    c4.timed(0, 1), 1, 128 * 2 * n4)
                del c4
            # C3: ER-500, 4096 episodes per GPU (32 768 at 8 GPUs), T = 1000, sharded, best cuts all-gathered
            n3 = 500
            c3 = Rollout(er_graphs(64, n3, 0.15, seed=10 + rank), 4096, 2 * n3, wd, seed=30 + rank)
            c3.step(n_steps=20)
            side["c3_er500"] = c3.side_block("ER_500spin (p=0.15, +-1), configs[2]: 4096 episodes per GPU over 64 graphs per GPU, "
                                             "2N = 1000 steps, episodes sharded, best cuts all-gathered",
                                             c3.timed(0, 1), 1, 4096 * 2 * n3, ranks=world)
            del c3
        except Exception as e:              # a side block must not cost the bench line
            side["sizes_error"] = "%s: %s" % (type(e).__name__, e)

    dqn = None
    if not args.skip_dqn:
        try:
            dqn = dqn_update_sample()
        except Exception as e:
            dqn = {"error": "%s: %s" % (type(e).__name__, e)}

    if rank == 0:
        avg_mpnn_s = r["mpnn_ms"] / 1000.0
        ach = flops_mpnn(n) * B / avg_mpnn_s / 1e12
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if head.used_impl == "tcgen05" and os.path.exists(tpath):      # dram bytes per launch from the committed ncu capture
            tj = json.load(open(tpath))["mpnn_tc_kernel"]
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj.get("source")
        # one-launch rollout: a launch covers T steps of [forward + argmax + env step]; traffic / bytes are per STEP
        spl = T if r["one_launch"] else 1
        roof = {"bound": "tensor",
                "kernel": ("mpnn_tc_kernel, one launch per rollout: T x (forward + argmax + env step)" if r["one_launch"]
                           else "mpnn_forward_argmax (%s)" % head.used_impl),
                "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": ach / pk["tflops"],
                "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes": int(B * (n * n + 3 * n * 4 + 16 + n * 4 + 4)),     # int8 J + features + degrees + action
                "traffic_and_bytes_are": "per rollout step (one forward over the batch)",
                "peak_source": pk["source"] + " (bf16 sustained)", "avg_launch_ms": avg_mpnn_s * 1e3 * spl,
                "steps_per_launch": spl, "ms_per_forward": avg_mpnn_s * 1e3,
                "launches_timed": r["mpnn_n"] // spl, "launches": T * args.steps // spl,
                "share_of_step": avg_mpnn_s * 1e3 * T * args.steps / ms_total,
                "flops_per_launch": flops_mpnn(n) * B * spl}
        avg_env_s, env_n = (r["env_ms"] / 1000.0, r["env_n"]) if not r["one_launch"] else (env_small[0] / 1000.0, env_small[1])
        roof_env = {"bound": "hbm", "kernel": "env_step", "achieved": bytes_env(n) * B / avg_env_s / 1e9,
                    "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": bytes_env(n) * B / avg_env_s / 1e9 / pk["hbm_gbs"],
                    "avg_launch_us": avg_env_s * 1e6, "launches_timed": env_n,
                    "share_of_step": None if r["one_launch"] else avg_env_s * 1e3 * T * args.steps / ms_total,
                    "note": ("the env-step kernel launched alone at the bench's batch (inside the rollout the step is applied by "
                             "the MPNN kernel's tail warp); " if r["one_launch"] else "") +
                            "B=4096 moves only %.1f MB per launch: launch-latency bound; see env_only" %
                            (bytes_env(n) * B / 1e6)}
        cpu = None
        if not args.skip_cpu and world == 1:          # side numbers: rank 0 at N = 1 only (the other ranks would wait)
            ref = CpuReference()
            ref.warm(J[0], wd)
            n_eps, sf = CPU_SAMPLE
            v, secs = ref.run(J[0], wd, n_eps, sf)
            cpu = {"value": v, "unit": "env-steps/s", "cores": ref.cores, "kind": ref.kind,
                   "sample": ref.describe(n_eps, sf, n, secs)}
        line = {"metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16x2-split/f32" if head.used_impl == "tcgen05" else "f32",
                "data": "synthetic", "config": headline_config(world),
                "e2e": {"value": e2e_value, "unit": "env-steps/s",
                        "h2d_bytes_per_step": int(G * n * n + B * 4 + B * n), "d2h_bytes_per_step": int(B * 4 + B * n),
                        "steps": e2e_steps},
                "gpu_launches": r["launches"], "roofline": roof, "roofline_env_step": roof_env, "env_only": env_only,
                "cpu_baseline": cpu, "clocks": r["clocks"], "mpnn_impl": head.used_impl,
                "mean_best_cut": float(bc.float().mean().item()), "c5_dqn": dqn}
        line.update(side)
        print(json.dumps(line))
    if world > 1:
        # every rank leaves together; a hard exit instead of destroy_process_group(), which can block while a captured
        # update (CUDA graph) still references the communicator
        sys.stdout.flush()
        dist.barrier()
        torch.cuda.synchronize()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mpnn", default="auto", choices=["auto", "simt", "tc"])
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-env-only", action="store_true")
    ap.add_argument("--skip-dqn", action="store_true")
    ap.add_argument("--skip-sizes", action="store_true", help="omit the side blocks c1 .. c4")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the headline workload returned on rank 0 (best_cut [B], "
                         "best_spins [B, N], steps [B]; 6.6 MB) as DIR/<name>.npy in float64; the inputs are seeded, so "
                         "two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the CUDA arm (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
