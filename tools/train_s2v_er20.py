"""Evidence that DQN.learn trains S2V-DQN agents: irreversible spins starting at -1, spin-only observation, dense reward,
MPNN(n_obs_in=1) (the reference's S2V recipe: dqn.py with reversible_spins=False, train_eco.py:311-315), on ER-20 (p = 0.15,
+-1), max_steps = N, acting with 16 lock-step environments on the device.  Hyper-parameters: those of tools/train_er20.py (the
reference's ER-20 ECO recipe, train_eco.py:114-161) with the episode length N -- minibatch 64, update every 32 timesteps,
target sync 1000, replay 5000, epsilon 1 -> 0.05 over 150 000 steps, lr 1e-4, gamma 0.95, Double-DQN, MSE, test every
10 000 timesteps with TestMetric.BEST.  Test set: the 16 ER-20 validation graphs of tests/golden/graphsets.npz (optimal cuts
known), one greedy-Q episode per graph from all -1 per evaluation.

A last line times the S2V trainer at ER-40 the way bench.py `c5_dqn` times the ECO trainer (minibatch 64, update every 32
timesteps, 16 lock-step environments, host clock around synchronised calls), with the ECO trainer measured in the same process.

    python tools/train_s2v_er20.py [timesteps=300000]  > profiles/r03_training_curve_s2v_er20.txt
"""
import os
import pickle
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import eco_dqn_b200.envs.core as ising_env  # noqa: E402
from eco_dqn_b200.envs.utils import (DEFAULT_OBSERVABLES, Observable, RewardSignal, ExtraAction, OptimisationTarget,  # noqa: E402
                                     SpinBasis, Stopping, RandomErdosRenyiGraphGenerator, SetGraphGenerator, EdgeType)
from eco_dqn_b200.networks.mpnn import MPNN  # noqa: E402
from eco_dqn_b200.agents.dqn.dqn import DQN  # noqa: E402
from eco_dqn_b200.agents.dqn.utils import TestMetric  # noqa: E402

HYPER = dict(init_weight_std=0.01, double_dqn=True, clip_Q_targets=False, gamma=0.95, replay_start_size=500,
             replay_buffer_size=5000, update_target_frequency=1000, update_learning_rate=False, initial_learning_rate=1e-4,
             peak_learning_rate=1e-4, peak_learning_rate_step=20000, final_learning_rate=1e-4, final_learning_rate_step=200000,
             update_frequency=32, minibatch_size=64, max_grad_norm=None, weight_decay=0, update_exploration=True,
             initial_exploration_rate=1, final_exploration_rate=0.05, final_exploration_step=150000, adam_epsilon=1e-8,
             logging=False, loss="mse", save_network_frequency=10 ** 9, test_frequency=10000, test_metric=TestMetric.BEST,
             n_envs=16)
S2V_ENV = {'observables': [Observable.SPIN_STATE], 'reward_signal': RewardSignal.DENSE, 'extra_action': ExtraAction.NONE,
           'optimisation_target': OptimisationTarget.CUT, 'spin_basis': SpinBasis.SIGNED, 'norm_rewards': True,
           'memory_length': None, 'horizon_length': None, 'stag_punishment': None, 'basin_reward': None,
           'reversible_spins': False}


def eco_env(n):
    return {'observables': DEFAULT_OBSERVABLES, 'reward_signal': RewardSignal.BLS, 'extra_action': ExtraAction.NONE,
            'optimisation_target': OptimisationTarget.CUT, 'spin_basis': SpinBasis.SIGNED, 'norm_rewards': True,
            'memory_length': None, 'horizon_length': None, 'stag_punishment': None, 'basin_reward': 1. / n,
            'reversible_spins': True, 'stopping': Stopping.NORMAL}


def quiet(f):
    with open(os.devnull, "w") as dn:
        old, sys.stdout = sys.stdout, dn
        try:
            return f()
        finally:
            sys.stdout = old


def time_er40(s2v, timesteps=3000):
    """ms per train_step and per 1000 timesteps of DQN.learn at ER-40 (bench.py dqn_update_sample's method)."""
    n = 40
    args = S2V_ENV if s2v else eco_env(n)
    env = ising_env.make("SpinSystem", RandomErdosRenyiGraphGenerator(n, 0.15, EdgeType.DISCRETE), n if s2v else 2 * n, **args)
    tmp = tempfile.mkdtemp()
    agent = DQN([env], (lambda: MPNN(n_obs_in=1)) if s2v else (lambda: MPNN()), init_weight_std=0.01, double_dqn=True,
                gamma=0.95, update_learning_rate=False, initial_learning_rate=1e-4, minibatch_size=64, update_frequency=32,
                update_target_frequency=1000, replay_start_size=500, replay_buffer_size=5000, final_exploration_step=3000,
                final_exploration_rate=0.05, test_frequency=10 ** 9, save_network_frequency=10 ** 9, logging=False, seed=5,
                test_metric=TestMetric.BEST, test_save_path=os.path.join(tmp, "s"), network_save_path=os.path.join(tmp, "n"),
                n_envs=16)
    acc = {"s": 0.0, "n": 0}
    orig = agent._train_step_device

    def timed(tr):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = orig(tr)
        torch.cuda.synchronize()
        acc["s"] += time.perf_counter() - t0
        acc["n"] += 1
        return out

    agent._train_step_device = timed
    quiet(lambda: agent.learn(timesteps=1000))
    acc["s"], acc["n"] = 0.0, 0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    quiet(lambda: agent.learn(timesteps=timesteps))
    torch.cuda.synchronize()
    return acc["s"] / max(acc["n"], 1) * 1e3, (time.perf_counter() - t0) / timesteps * 1e6


def main():
    steps = int(sys.argv[1]) if len(sys.argv) > 1 else 300000
    n = 20
    gs = np.load(os.path.join(ROOT, "tests", "golden", "graphsets.npz"))
    test_graphs = [g.astype(np.float64) for g in gs["er20"]]
    opt = gs["er20_opt"].astype(np.float64)
    train_env = ising_env.make("SpinSystem", RandomErdosRenyiGraphGenerator(n, 0.15, EdgeType.DISCRETE), n, **S2V_ENV)
    test_env = ising_env.make("SpinSystem", SetGraphGenerator(test_graphs, ordered=True), n, **S2V_ENV)
    tmp = tempfile.mkdtemp()
    agent = DQN([train_env], lambda: MPNN(n_obs_in=1), network_save_path=os.path.join(tmp, "net"), evaluate=True,
                test_envs=[test_env], test_episodes=len(test_graphs), test_save_path=os.path.join(tmp, "scores"), seed=1,
                **HYPER)
    untrained = agent.evaluate_agent()[1]
    torch.cuda.synchronize()
    t0 = time.time()
    quiet(lambda: agent.learn(timesteps=steps))
    torch.cuda.synchronize()
    wall = time.time() - t0
    with open(os.path.join(tmp, "solution.pkl"), "rb") as f:
        curve = pickle.load(f)
    try:
        import subprocess
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception:
        gpu = torch.cuda.get_device_properties(0).name
    print("# S2V-DQN on ER-20, max_steps = N, %d timesteps in %.1f s on one GPU (%s) (%.1f us per timestep incl. %d evaluations)"
          % (steps, wall, gpu, wall / steps * 1e6, len(curve)))
    print("# mean optimal cut of the 16 test graphs: %.3f; untrained network (greedy-Q from all -1): %.3f" % (opt.mean(), untrained))
    print("# timestep  mean_best_cut  ratio_to_optimal")
    for ts, sol in curve:
        print("%9d  %8.3f  %6.3f" % (ts, sol, sol / opt.mean()))
    tail = np.array([s for _, s in curve[-10:]])
    print("# mean of the last 10 evaluations: %.3f = %.3f of optimal" % (tail.mean(), tail.mean() / opt.mean()))
    s2v = time_er40(True)
    eco = time_er40(False)
    print("# ER-40, 16 lock-step environments, minibatch 64, update every 32 timesteps (bench.py c5_dqn method), same process: "
          "S2V-DQN train_step %.3f ms, %.1f ms per 1000 timesteps; ECO-DQN train_step %.3f ms, %.1f ms per 1000 timesteps"
          % (s2v[0], s2v[1], eco[0], eco[1]))
    sys.stdout.flush()
    assert tail.mean() >= 0.90 * opt.mean() and tail.mean() > untrained, "the agent did not learn"


if __name__ == "__main__":
    main()
