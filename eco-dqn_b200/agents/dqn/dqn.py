"""Double-DQN trainer on the batched device engine (reference src/agents/dqn/dqn.py:20-610, BASELINE config 5).

Same constructor keywords, same update rule (dqn.py:403-451: Double-DQN target, MSE / Huber, Adam, optional
gradient clipping), same schedules (dqn.py:467-487), same evaluation metric and checkpoint format (dqn.py:604-610,
`torch.save(state_dict)`).  What changes is where the work runs:

  * acting: `n_envs` episodes step in lock-step on the device (n_envs = 1 is the reference's schedule); the greedy
    branch is the fused MPNN + argmax kernel, evaluated per environment like the reference's B = 1 forward;
  * replay: compact device-resident transitions (agents/dqn/utils.py) pointing into a device ring of graphs;
  * update: target Q-values come from the CUDA forward kernels; loss and all 12 gradient tensors come from the
    hand-written forward/backward kernels (eco_mpnn_grad) and Adam is one kernel (eco_mpnn_adam).  Only a
    user-supplied loss callable takes the autograd route through the PyTorch module.  With several ranks the
    gradients are averaged with ONE all-reduce over the flat gradient buffer (NCCL over NVLink), then every rank
    applies the same Adam step.

Differences from the reference that a caller can see: `test_metric` defaults to TestMetric.BEST (the reference's
default ENERGY_ERROR has no branch left in its evaluate_agent and always scores 0); BEST and FINAL are supported.
`logging` is accepted and ignored (the reference's pickle Logger is out of scope; every script passes False).
"""
import os
import pickle
import random
import time

import numpy as np
import torch
import torch.nn.functional as F
import torch.optim as optim

from ... import engine, sharding
from ... import _lib
from ..._lib import lib, check
from .utils import KernelAdam, ReplayBuffer, TestMetric, set_global_seed
from ...envs.utils import OptimisationTarget

import ctypes as C


class DQN:
    def __init__(self, envs, network, init_network_params=None, init_weight_std=None, double_dqn=True,
                 update_target_frequency=10000, gamma=0.99, clip_Q_targets=False, replay_start_size=50000,
                 replay_buffer_size=1000000, minibatch_size=32, update_frequency=1, update_learning_rate=True,
                 initial_learning_rate=0, peak_learning_rate=1e-3, peak_learning_rate_step=10000,
                 final_learning_rate=5e-5, final_learning_rate_step=200000, max_grad_norm=None, weight_decay=0,
                 update_exploration=True, initial_exploration_rate=1, final_exploration_rate=0.1,
                 final_exploration_step=1000000, adam_epsilon=1e-8, loss="mse", save_network_frequency=10000,
                 network_save_path='network', evaluate=True, test_envs=None, test_episodes=20, test_frequency=10000,
                 test_save_path='test_scores', test_metric=TestMetric.BEST, logging=True, seed=None, n_envs=1,
                 dp_mode="peer", cuda_graph=True):
        self.device = engine._require_cuda()
        self.rank, self.world = sharding.world_info()
        self.double_dqn = double_dqn
        self.replay_start_size = replay_start_size
        self.replay_buffer_size = replay_buffer_size
        self.gamma = gamma
        self.clip_Q_targets = clip_Q_targets
        self.update_target_frequency = update_target_frequency
        self.minibatch_size = minibatch_size
        self.update_learning_rate = update_learning_rate
        self.initial_learning_rate = initial_learning_rate
        self.peak_learning_rate = peak_learning_rate
        self.peak_learning_rate_step = peak_learning_rate_step
        self.final_learning_rate = final_learning_rate
        self.final_learning_rate_step = final_learning_rate_step
        self.max_grad_norm = max_grad_norm
        self.weight_decay = weight_decay
        self.update_frequency = update_frequency
        self.update_exploration = True        # the reference stores a 1-tuple here, which is always truthy (dqn.py:161)
        self.initial_exploration_rate = initial_exploration_rate
        self.epsilon = self.initial_exploration_rate
        self.final_exploration_rate = final_exploration_rate
        self.final_exploration_step = final_exploration_step
        self.adam_epsilon = adam_epsilon
        self.logging = logging
        self._loss_kind = None                # ECO_LOSS_* when the gradient kernels can take the loss
        self._grad_scratch = None
        if dp_mode not in ("peer", "nccl"):
            raise ValueError("dp_mode must be 'peer' (gradient exchange over CUDA IPC peer memory, fused with Adam) or 'nccl'")
        self.dp_mode = dp_mode                # how the ranks' gradients are averaged (world > 1)
        self.cuda_graph = bool(cuda_graph)    # replay the update (TD target .. Adam .. re-pack) as one CUDA graph
        self.overlap_target = os.environ.get("ECO_DQN_OVERLAP_TARGET", "1") != "0"   # TD target on a second stream (see _update)
        self._ag = None                       # the captured acting step (n_envs > 1), see _capture_act
        self._tgt_stream = None
        self._cg = None
        if callable(loss):
            self.loss = loss
        else:
            try:
                self.loss = {'huber': F.smooth_l1_loss, 'mse': F.mse_loss}[loss]
                self._loss_kind = {'mse': _lib.LOSS_MSE, 'huber': _lib.LOSS_HUBER}[loss]
            except KeyError:
                raise ValueError("loss must be 'huber', 'mse' or a callable")
        if test_metric not in (TestMetric.BEST, TestMetric.FINAL):
            raise NotImplementedError("test_metric=%s: only TestMetric.BEST (default here) and TestMetric.FINAL are "
                                      "evaluated on this path" % (test_metric,))

        if type(envs) != list:
            envs = [envs]
        self.envs = envs
        self._check_uniform(envs, "training")
        if any(not e.reversible_spins for e in envs):
            raise NotImplementedError("irreversible (S2V-DQN) environments are outside the accelerated path")
        self.acting_in_reversible_spin_env = True
        self.n_spins, self.max_steps = envs[0].n_spins, envs[0].max_steps
        self.basin_reward = envs[0].basin_reward
        self.min_cut = envs[0].optimisation_target == OptimisationTarget.MIN_CUT
        self.n_envs = int(n_envs)

        self.seed = random.randint(0, int(1e6)) if seed is None else seed      # dqn.py:187 (int() for Python 3.12)
        set_global_seed(self.seed + self.rank)
        self._gen = torch.Generator(device=self.device)
        self._gen.manual_seed(self.seed + 7919 * self.rank)

        self.network = network().to(self.device)
        self.init_network_params = init_network_params
        self.init_weight_std = init_weight_std
        if init_network_params is not None:
            self.load(init_network_params)
        elif init_weight_std is not None:
            with torch.no_grad():
                for m in self.network.modules():
                    if type(m) == torch.nn.Linear:
                        m.weight.normal_(0, init_weight_std)
        if self.world > 1:                       # every rank starts from rank 0's parameters
            for p in self.network.parameters():
                torch.distributed.broadcast(p.data, src=0)
        self.target_network = network().to(self.device)
        self.target_network.load_state_dict(self.network.state_dict())
        for p in self.target_network.parameters():
            p.requires_grad = False
        if self.network.engine_weights(self.device).aliases:
            # Adam in one hand-written kernel over the live parameters (eco_mpnn_adam)
            self.optimizer = KernelAdam(self.network, lr=self.initial_learning_rate, eps=self.adam_epsilon,
                                        weight_decay=self.weight_decay)
        else:
            self.optimizer = optim.Adam(self.network.parameters(), lr=self.initial_learning_rate, eps=self.adam_epsilon,
                                        weight_decay=self.weight_decay)

        self.evaluate = evaluate
        if test_envs in [None, [None]]:
            self.test_envs = self.envs
        else:
            self.test_envs = test_envs if type(test_envs) == list else [test_envs]
        self._check_uniform(self.test_envs, "test")
        if any(not e.reversible_spins for e in self.test_envs):
            raise NotImplementedError("irreversible (S2V-DQN) environments are outside the accelerated path")
        self.test_episodes = int(test_episodes)
        self.test_frequency = test_frequency
        self.test_save_path = test_save_path
        self.test_metric = test_metric
        self.losses_save_path = os.path.join(os.path.split(self.test_save_path)[0], "losses.pkl")
        self.solution_save_path = os.path.join(os.path.split(self.test_save_path)[0], "solution.pkl")
        self.allowed_action_state = (-1, 1)
        self.save_network_frequency = save_network_frequency
        self.network_save_path = network_save_path

        # ---- device state: graph ring, lock-step environments, replay --------------------------------------
        n, T, E = self.n_spins, self.max_steps, self.n_envs
        self._ring_size = int(np.ceil(replay_buffer_size / T)) + 2 * E + 2
        first = [self._new_graph() for _ in range(E)]
        if not all(engine.is_int8_graph(g) for g in first):
            raise NotImplementedError("DQN training with real-valued couplings (EdgeType.RANDOM) is not supported: the "
                                      "training kernels take integer couplings; weighted graphs run rollouts only")
        if n > _lib.MAX_SPINS:
            raise NotImplementedError("DQN training on graphs of more than %d vertices is not supported: the training kernels "
                                      "take the dense layout; sparse (CSR) graph sets run rollouts only" % _lib.MAX_SPINS)
        ring = np.zeros((self._ring_size, n, n), dtype=np.int8)
        ring[:] = engine.graphs_to_int8(first[0])[0]          # placeholder so that every slot holds a valid graph
        self._graphs = engine.GraphSet(ring, device=self.device, min_cut=self.min_cut)
        self._ring_pos = 0
        self._env = engine.BatchedSpinSystem(self._graphs, E, T, self.basin_reward)
        self.replay_buffer = ReplayBuffer(replay_buffer_size, self._env.NP, self.device)
        self.replay_buffers = {n: self.replay_buffer}
        self._start_episodes(first)
        # the update's batch normaliser (mpnn.py:102: the largest degree in the minibatch) stays on the device: the kernels
        # read `*dmax` of the graph set they are given when norm_max == 0, so the update passes a copy of the graph-set
        # struct whose dmax points at a one-float buffer it fills itself
        self._nm_buf = torch.ones(1, dtype=torch.float32, device=self.device)
        self._graphs_nm = type(self._graphs.c)()
        C.memmove(C.byref(self._graphs_nm), C.byref(self._graphs.c), C.sizeof(self._graphs_nm))
        self._graphs_nm.dmax = self._nm_buf.data_ptr()
        self._fused_dp = False
        if self.world > 1 and isinstance(self.optimizer, KernelAdam):
            if self.dp_mode == "peer" and self.max_grad_norm is None:
                def gather(mine):
                    out = [torch.zeros(64, dtype=torch.uint8, device=self.device) for _ in range(self.world)]
                    torch.distributed.all_gather(out, mine.to(self.device))
                    return torch.stack(out)
                self.optimizer.attach_peers(self.world, self.rank, gather)
                self._fused_dp = True
            else:
                self.optimizer.grad_scale = 1.0 / self.world       # SUM all-reduce, the mean is taken inside the Adam kernel

    # ------------------------------------------------------------------ environment plumbing
    @staticmethod
    def _check_uniform(envs, what):
        """One device batch steps every environment of a list: they must agree on what the kernels are configured with."""
        for attr in ("n_spins", "max_steps", "optimisation_target", "basin_reward", "reversible_spins"):
            if len(set(getattr(e, attr) for e in envs)) != 1:
                raise NotImplementedError("all %s environments must share %s (got %s)" %
                                          (what, attr, sorted(set(str(getattr(e, attr)) for e in envs))))

    def _new_graph(self):
        env = random.sample(self.envs, k=1)[0]                # get_random_env, dqn.py:242-248
        return np.asarray(env.gg.get())

    def _write_ring(self, graphs):
        """Put `graphs` into consecutive ring slots (wrapping) and return the slot indices."""
        E = len(graphs)
        slots = [(self._ring_pos + i) % self._ring_size for i in range(E)]
        self._ring_pos = (self._ring_pos + E) % self._ring_size
        J = torch.from_numpy(engine.graphs_to_int8(np.stack(graphs))).to(self.device)
        start = 0
        while start < E:                                      # contiguous runs (at most two: the ring wraps once)
            run = 1
            while start + run < E and slots[start + run] == slots[start + run - 1] + 1:
                run += 1
            check(lib().eco_graphs_update(C.byref(self._graphs.c), slots[start], run,
                                          C.c_void_p(J[start:start + run].contiguous().data_ptr()), engine._stream()))
            start += run
        torch.cuda.current_stream().synchronize()
        flags = self._graphs.gstat[torch.tensor(slots, device=self.device), 3].cpu().numpy()
        if (flags & 7).any():
            raise NotImplementedError("training graphs must be symmetric, non-empty, with couplings in {-1,0,1}")
        return np.array(slots, dtype=np.int32)

    def _start_episodes(self, graphs=None):
        E = self.n_envs
        if graphs is None:
            graphs = [self._new_graph() for _ in range(E)]
        slots = self._write_ring(graphs)
        spins = np.stack([2 * np.random.randint(2, size=self.n_spins) - 1 for _ in range(E)])   # spinsystem.py:294
        self._env.reset(spins=spins, graph_idx=slots)
        if getattr(self, "_scores", None) is None:
            self._scores = torch.zeros(E, dtype=torch.float64, device=self.device)
        else:
            self._scores.zero_()          # (in place: the captured acting step holds its address)

    def _obs_from(self, xn, xg, graph):
        """[B, 7 + N, N] fp32 observations in the reference's layout, rebuilt on the device for the autograd forward."""
        n = self.n_spins
        rows = torch.cat([xn[:, :, :n], xg.unsqueeze(-1).expand(-1, -1, n)], dim=1)
        adj = self._graphs.J[graph.long(), :n, :n].to(torch.float32)
        return torch.cat([rows, adj], dim=1)

    def _q_kernel(self, network, xn, xg, graph, norm_max, want_q=True, graphs_c=None):
        """Q-values / argmax through the CUDA forward kernels for arbitrary (replayed) features."""
        graphs_c = self._graphs.c if graphs_c is None else graphs_c
        B = xn.shape[0]
        w = network.engine_weights(self.device)
        q = torch.zeros(B, self._env.NP, dtype=torch.float32, device=self.device) if want_q else None
        act = torch.zeros(B, dtype=torch.int32, device=self.device)
        scratch = self._env._scratch_for(B)
        xn, xg, graph = xn.contiguous(), xg.contiguous(), graph.to(torch.int32).contiguous()
        check(lib().eco_mpnn_forward(C.byref(graphs_c), C.byref(w.c), B, engine._ptr(graph), engine._ptr(xn),
                                     engine._ptr(xg), float(norm_max), engine._ptr(q), engine._ptr(act),
                                     engine._ptr(scratch), self._env.mpnn_impl, engine._stream()))
        return (q[:, :self.n_spins] if want_q else None), act

    # ------------------------------------------------------------------ learning
    def learn(self, timesteps, verbose=False):
        E = self.n_envs
        env = self._env
        losses, test_scores, test_solutions, losses_eps = [], [], [], []
        is_training_ready = False
        t1 = time.time()
        timestep = 0
        while timestep < timesteps:
            if not is_training_ready and len(self.replay_buffer) >= self.replay_start_size:
                print('\nAll buffers have {} transitions stored - training is starting!\n'.format(self.replay_start_size))
                is_training_ready = True

            if self._act_graph_ok():
                # several lock-step environments: act -> step -> replay append as ONE captured graph (see _capture_act)
                self._act_step_graph(timestep, is_training_ready)
                if self.update_learning_rate:
                    self.update_lr(timestep)
            else:
                xn, xg, graph = env.xn.clone(), env.xg.clone(), env.graph_idx.clone()
                actions = self.act((xn, xg, graph), is_training_ready)
                if self.update_exploration:
                    self.update_epsilon(timestep)
                if self.update_learning_rate:
                    self.update_lr(timestep)
                reward, done = env.step(actions)
                self._scores += reward
                self.replay_buffer.add(xn, xg, actions, reward, env.xn, env.xg, done, graph)
            t_before, timestep = timestep, timestep + E

            if env.current_step == self.max_steps:            # lock-step: every episode ends together
                if verbose:
                    losses_eps = [float(x) for x in losses_eps]
                    loss_str = "{:.2e}".format(np.mean(losses_eps)) if (is_training_ready and losses_eps) else "N/A"
                    print("timestep : {}, episode time: {}, score : {}, mean loss: {}, time : {} s".format(
                        timestep, env.current_step, np.round(float(self._scores.mean()), 3), loss_str,
                        round(time.time() - t1, 3)))
                self._start_episodes()
                losses_eps = []
                t1 = time.time()

            if is_training_ready:
                for _ in range(self._crossings(t_before, timestep, self.update_frequency)):
                    # (the loss stays on the device: one host read per episode / at the end instead of one per update)
                    loss = self._train_step_device(self.replay_buffer.sample_indices(self.minibatch_size, self._gen))
                    losses.append([timestep, loss])
                    losses_eps.append(loss)
                if self._crossings(t_before, timestep, self.update_target_frequency):
                    self.target_network.load_state_dict(self.network.state_dict())
                    self.target_network.engine_weights(self.device)      # re-pack now: a replayed graph would not

            if self._crossings(t_before + 1, timestep + 1, self.test_frequency) and self.evaluate and is_training_ready:
                test_score, test_solution = self.evaluate_agent()
                print('\nTest score: {}\nTest solution: {}\n'.format(np.round(test_score, 3), np.round(test_solution, 3)))
                if all(test_score > s for _, s in test_scores) and self.rank == 0:
                    main, ext = os.path.splitext(self.network_save_path)
                    self.save(main + "_best" + (ext if ext else '.pth'))
                test_scores.append([timestep, test_score])
                test_solutions.append([timestep, test_solution])
            if self._crossings(t_before + 1, timestep + 1, self.save_network_frequency) and is_training_ready \
                    and self.rank == 0:
                main, ext = os.path.splitext(self.network_save_path)
                self.save(main + str(timestep) + (ext if ext else '.pth'))

        if losses and torch.is_tensor(losses[0][1]):          # one device -> host copy for all the recorded losses
            vals = torch.stack([l for _, l in losses]).reshape(-1).cpu().tolist()
            losses = [[ts, v] for (ts, _), v in zip(losses, vals)]
        if self.rank == 0:
            path = self.test_save_path if os.path.splitext(self.test_save_path)[-1] else self.test_save_path + '.pkl'
            for p, obj in ((path, test_scores), (self.losses_save_path, losses), (self.solution_save_path, test_solutions)):
                if os.path.dirname(p):
                    os.makedirs(os.path.dirname(p), exist_ok=True)
                with open(p, 'wb+') as output:
                    pickle.dump(np.array(obj), output, pickle.HIGHEST_PROTOCOL)
        return losses

    @staticmethod
    def _crossings(t0, t1, period):
        """How many multiples of `period` lie in [t0, t1): the reference tests `timestep % period == 0` once per step."""
        if period <= 0:
            return 0
        return (t1 + period - 1) // period - (t0 + period - 1) // period

    def train_step(self, transitions):
        """reference dqn.py:403-451 on a dict of compact transitions (see ReplayBuffer.FIELDS); returns the loss as a float
        like the reference (one host read: `learn` uses the device-side form below instead)."""
        return float(self._update(transitions))

    def _update(self, t):
        """One update entirely on the device -- no host read: Double-DQN target through the forward kernels, loss and
        gradients through eco_mpnn_grad, gradient mean over ranks + Adam (+ re-pack).  Returns the loss as a device tensor."""
        graph = t["graph"]
        if self._loss_kind is None:
            return self._update_autograd(t)
        with torch.no_grad():
            # the reference feeds the whole minibatch through the network: norm.max() is the batch's max degree
            self._nm_buf.copy_(self._graphs.gstat[graph.long(), 0].max().clamp(min=1).to(torch.float32).reshape(1))
            gc = self._graphs_nm                       # norm_max = 0 -> the kernels read *dmax = _nm_buf

            def td_target_of():
                if self.double_dqn:
                    _, greedy = self._q_kernel(self.network, t["xn_next"], t["xg_next"], graph, 0.0, want_q=False, graphs_c=gc)
                    q_tgt, _ = self._q_kernel(self.target_network, t["xn_next"], t["xg_next"], graph, 0.0, graphs_c=gc)
                    q_value_target = q_tgt.gather(1, greedy.long().unsqueeze(1))
                else:
                    q_tgt, _ = self._q_kernel(self.target_network, t["xn_next"], t["xg_next"], graph, 0.0, graphs_c=gc)
                    q_value_target = q_tgt.max(1, True)[0]
                if self.clip_Q_targets:
                    q_value_target = q_value_target.clamp(min=0)
                return t["reward"].unsqueeze(1) + (1 - t["done"].unsqueeze(1)) * self.gamma * q_value_target

            # forward + backward of the online network in the hand-written kernels (eco_mpnn_grad, csrc/mpnn_grad.cu).  Its
            # forward pass does not need the regression targets: the Double-DQN target (two forwards of the next states +
            # a handful of small tensor ops) runs on a second stream underneath it and is waited for just before the readout
            # (eco_mpnn_grad_ev); in the captured update the two branches are parallel paths of the CUDA graph.
            if self.overlap_target:
                main = torch.cuda.current_stream()
                if self._tgt_stream is None:
                    self._tgt_stream = torch.cuda.Stream(device=self.device)
                self._tgt_stream.wait_stream(main)
                with torch.cuda.stream(self._tgt_stream):
                    td_target = td_target_of().reshape(-1).to(torch.float32).contiguous()
                    ready = torch.cuda.Event()
                    ready.record(self._tgt_stream)
                td_target.record_stream(main)
                loss = self._grad_kernel(t["xn"], t["xg"], graph, 0.0, t["action"], td_target, graphs_c=gc, ready=ready)
            else:
                loss = self._grad_kernel(t["xn"], t["xg"], graph, 0.0, t["action"], td_target_of(), graphs_c=gc)
            if self.world > 1 and not self._fused_dp:
                self._allreduce_grads()
            if self.max_grad_norm is not None:
                torch.nn.utils.clip_grad_norm_(self.network.parameters(), self.max_grad_norm)
            self.optimizer.step()
        return loss

    def _update_autograd(self, t):
        """A user-supplied loss callable: autograd through the PyTorch module (networks/mpnn.py::forward); its gradients
        feed the same Adam kernel."""
        graph = t["graph"]
        with torch.no_grad():
            norm_max = float(self._graphs.gstat[graph.long(), 0].max().clamp(min=1).item())
            if self.double_dqn:
                _, greedy = self._q_kernel(self.network, t["xn_next"], t["xg_next"], graph, norm_max, want_q=False)
                q_tgt, _ = self._q_kernel(self.target_network, t["xn_next"], t["xg_next"], graph, norm_max)
                q_value_target = q_tgt.gather(1, greedy.long().unsqueeze(1))
            else:
                q_tgt, _ = self._q_kernel(self.target_network, t["xn_next"], t["xg_next"], graph, norm_max)
                q_value_target = q_tgt.max(1, True)[0]
            if self.clip_Q_targets:
                q_value_target[q_value_target < 0] = 0
            td_target = t["reward"].unsqueeze(1) + (1 - t["done"].unsqueeze(1)) * self.gamma * q_value_target
        q_all = self.network(self._obs_from(t["xn"], t["xg"], graph))
        if q_all.dim() == 1:
            q_all = q_all.unsqueeze(0)
        q_value = q_all.gather(1, t["action"].unsqueeze(1))
        loss = self.loss(q_value, td_target, reduction='mean')
        self.optimizer.zero_grad()
        loss.backward()
        if self.world > 1:
            sharding.allreduce_mean_grads(self.network.parameters())
        if self.max_grad_norm is not None:
            torch.nn.utils.clip_grad_norm_(self.network.parameters(), self.max_grad_norm)
        if isinstance(self.optimizer, KernelAdam):
            scale, self.optimizer.grad_scale = self.optimizer.grad_scale, 1.0      # (already averaged)
            dp, self.optimizer._dp = self.optimizer._dp, None
            self.optimizer.step()
            self.optimizer.grad_scale, self.optimizer._dp = scale, dp
        else:
            self.optimizer.step()
        return loss.detach()

    def _train_step_device(self, idx):
        """The update for the replay rows `idx` (device int64 [minibatch]); with cuda_graph the captured update is replayed."""
        if self._loss_kind is None or not self.cuda_graph or not isinstance(self.optimizer, KernelAdam):
            return self._update(self.replay_buffer.gather(idx)).detach().reshape(())
        if self._cg is None:
            self._capture_update(idx)
        self._g_idx.copy_(idx)
        self.optimizer.sync_lr()
        self._cg.replay()
        return self._g_loss.clone().reshape(())

    def _capture_update(self, idx):
        """Capture `_update` on the rows of a static index buffer.  The two warm-up runs (allocations, lazy initialisation,
        NCCL channels) are real updates, so parameters and optimizer state are saved before and put back after."""
        opt = self.optimizer
        self._g_idx = idx.clone()
        saved = [p.detach().clone() for p in self.network.parameters()]
        state = (opt.exp_avg.clone(), opt.exp_avg_sq.clone(), opt.step_dev.clone())
        opt.sync_lr()
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self._update(self.replay_buffer.gather(self._g_idx))
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize(self.device)

        def restore():
            with torch.no_grad():
                for p, q in zip(self.network.parameters(), saved):
                    p.copy_(q)
                opt.exp_avg.copy_(state[0]); opt.exp_avg_sq.copy_(state[1]); opt.step_dev.copy_(state[2])
            self.network.engine_weights(self.device).repack()
        restore()
        if self.world > 1:
            torch.distributed.barrier()       # (the exchange epochs of eco_dp_adam count on their own: nothing to rewind)
        self._cg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._cg):
            self._g_loss = self._update(self.replay_buffer.gather(self._g_idx))
        torch.cuda.synchronize(self.device)

    def _grad_kernel(self, xn, xg, graph, norm_max, action, td_target, graphs_c=None, ready=None):
        """loss and d loss / d weights of the regression step (dqn.py:436-447) through eco_mpnn_grad; the gradient
        lands in `p.grad` of every parameter (views of one flat buffer, state_dict order)."""
        B = xn.shape[0]
        w = self.network.engine_weights(self.device)
        nb = lib().eco_mpnn_grad_scratch_bytes(B, self.n_spins)
        if self._grad_scratch is None or self._grad_scratch.numel() < nb:
            self._grad_scratch = torch.empty(nb, dtype=torch.uint8, device=self.device)
        flat = torch.empty(_lib.MPNN_N_PARAMS, dtype=torch.float32, device=self.device)
        loss = torch.empty(1, dtype=torch.float32, device=self.device)
        xn, xg, graph = xn.contiguous(), xg.contiguous(), graph.to(torch.int32).contiguous()
        action = action.to(torch.int32).contiguous()
        target = td_target.reshape(-1).to(torch.float32).contiguous()
        check(lib().eco_mpnn_grad_ev(C.byref(self._graphs.c if graphs_c is None else graphs_c), C.byref(w.c), B, engine._ptr(graph),
                                     engine._ptr(xn), engine._ptr(xg), float(norm_max), engine._ptr(action), engine._ptr(target),
                                     self._loss_kind, engine._ptr(loss), engine._ptr(flat), engine._ptr(self._grad_scratch),
                                     C.c_void_p(ready.cuda_event if ready is not None else 0), engine._stream()))
        params = dict(self.network.named_parameters())
        off = 0
        for key, shp in zip(engine.STATE_DICT_KEYS, engine.STATE_DICT_SHAPES):
            n = int(np.prod(shp))
            g = flat[off:off + n].view(shp)
            p = params[key]
            if tuple(p.shape) != shp:          # S2V-DQN nets (n_obs_in = 1): the kernels see zero-padded columns
                g = g[:, :p.shape[1]].contiguous()
            p.grad = g
            off += n
        return loss

    def _allreduce_grads(self):
        """dp_mode "nccl": one SUM all-reduce over the flat gradient buffer that eco_mpnn_grad wrote (the per-tensor
        gradients are views of it); the division by the world size is folded into the Adam kernel (grad_scale)."""
        flat = self.optimizer._flat_grad()
        torch.distributed.all_reduce(flat, op=torch.distributed.ReduceOp.SUM)

    # ------------------------------------------------------------------ captured acting step (n_envs > 1)
    def _act_graph_ok(self):
        return (self.cuda_graph and self.n_envs > 1 and self._loss_kind is not None and isinstance(self.optimizer, KernelAdam)
                and os.environ.get("ECO_DQN_ACT_GRAPH", "1") != "0")

    def _act_step_graph(self, timestep, is_training_ready):
        """One lock-step of `learn` for all environments -- snapshot of the observations, epsilon-greedy action (forward
        kernel + device draws), SpinSystemBase.step, score bookkeeping, replay append -- replayed as one CUDA graph: the
        eager form is ~25 small launches and ~0.4 ms of host time per lock-step for ~0.1 ms of device work.  Device-resident
        state: replay write position, exploration rate, the ready flag; the host keeps its mirrors (replay size, env step
        counter, epsilon) in step.  The device draws come from the agent's generator (registered with the graph)."""
        rb, env, E = self.replay_buffer, self._env, self.n_envs
        if self._ag is None:
            self._capture_act()
        self._ag_ready.fill_(bool(is_training_ready))
        self._ag_eps.fill_(float(self.epsilon))
        env._check_steppable()
        self._ag.replay()
        env.current_step += 1
        rb._position = (rb._position + E) % rb._capacity
        rb._size = min(rb._size + E, rb._capacity)
        if self.update_exploration:
            self.update_epsilon(timestep)

    def _act_body(self):
        rb, env, E, dev = self.replay_buffer, self._env, self.n_envs, self.device
        self._ag_xn.copy_(env.xn); self._ag_xg.copy_(env.xg); self._ag_graph.copy_(env.graph_idx)
        rand_actions = torch.randint(0, self.n_spins, (E,), device=dev, generator=self._gen, dtype=torch.int32)
        greedy = self._q_kernel(self.network, self._ag_xn, self._ag_xg, self._ag_graph, -1.0, want_q=False)[1]
        explore = torch.rand(E, device=dev, generator=self._gen) < self._ag_eps
        actions = torch.where(self._ag_ready & ~explore, greedy, rand_actions).contiguous()
        with torch.cuda.device(dev):
            check(lib().eco_env_step(C.byref(env.gs.c), C.byref(env.c), _lib.POLICY_ACTIONS, engine._ptr(actions),
                                     engine._ptr(env._reward), engine._ptr(env._done), None, None, None, engine._stream()))
        self._scores += env._reward
        idx = (self._ag_pos + torch.arange(E, device=dev)) % rb._capacity
        rb.xn[idx], rb.xg[idx] = self._ag_xn, self._ag_xg
        rb.xn_next[idx], rb.xg_next[idx] = env.xn, env.xg
        rb.action[idx] = actions.to(torch.int64)
        rb.reward[idx] = env._reward.to(torch.float32)
        rb.done[idx] = env._done.to(torch.float32)
        rb.graph[idx] = self._ag_graph
        self._ag_pos.add_(E).remainder_(rb._capacity)

    def _capture_act(self):
        rb, env, E, dev = self.replay_buffer, self._env, self.n_envs, self.device
        self._ag_xn, self._ag_xg, self._ag_graph = env.xn.clone(), env.xg.clone(), env.graph_idx.clone()
        self._ag_pos = torch.full((1,), rb._position, dtype=torch.int64, device=dev)
        self._ag_eps = torch.zeros(1, dtype=torch.float32, device=dev)
        self._ag_ready = torch.zeros(1, dtype=torch.bool, device=dev)
        # The warm-up run must leave no trace: it steps the environments and appends to the replay.  Save / restore the
        # environment workspace, the scores and the replay rows it touches.
        ws = env._ws.clone()
        scores = self._scores.clone()
        saved = {k: getattr(rb, k).clone() for k in rb.FIELDS}
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            self._act_body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize(dev)
        env._ws.copy_(ws); self._scores.copy_(scores)
        for k, v in saved.items():
            getattr(rb, k).copy_(v)
        self._ag_pos.fill_(rb._position)
        self._ag = torch.cuda.CUDAGraph()
        self._ag.register_generator_state(self._gen)
        with torch.cuda.graph(self._ag):
            self._act_body()

    def act(self, state, is_training_ready=True):
        """epsilon-greedy (reference dqn.py:453-465).  One environment: the reference's own draws, in its order
        (`random.uniform(0, 1) >= epsilon` -> greedy, else `np.random.randint(0, n)`), so a seeded run picks the
        reference's actions.  Several lock-step environments: one device draw per environment."""
        xn, xg, graph = state
        E = xn.shape[0]
        if E == 1:
            if is_training_ready and random.uniform(0, 1) >= self.epsilon:
                return self.predict(state)
            return torch.tensor([np.random.randint(0, self.n_spins)], dtype=torch.int32, device=self.device)
        rand_actions = torch.randint(0, self.n_spins, (E,), device=self.device, generator=self._gen, dtype=torch.int32)
        if not is_training_ready:
            return rand_actions
        greedy = self.predict(state)
        explore = torch.rand(E, device=self.device, generator=self._gen) < self.epsilon
        return torch.where(explore, rand_actions, greedy)

    @torch.no_grad()
    def predict(self, states, acting_in_reversible_spin_env=None):
        """argmax_a Q(s, a) per environment; every environment is normalised by its own graph, like the reference's
        one-environment forward (dqn.py:490-503)."""
        xn, xg, graph = states
        return self._q_kernel(self.network, xn, xg, graph, -1.0, want_q=False)[1]

    def update_epsilon(self, timestep):
        eps = self.initial_exploration_rate - (self.initial_exploration_rate - self.final_exploration_rate) * (
            timestep / self.final_exploration_step)
        self.epsilon = max(eps, self.final_exploration_rate)

    def update_lr(self, timestep):
        if timestep <= self.peak_learning_rate_step:
            lr = self.initial_learning_rate - (self.initial_learning_rate - self.peak_learning_rate) * (
                timestep / self.peak_learning_rate_step)
        elif timestep <= self.final_learning_rate_step:
            lr = self.peak_learning_rate - (self.peak_learning_rate - self.final_learning_rate) * (
                (timestep - self.peak_learning_rate_step) / (self.final_learning_rate_step - self.peak_learning_rate_step))
        else:
            lr = None
        if lr is not None:
            for g in self.optimizer.param_groups:
                g['lr'] = lr

    @torch.no_grad()
    def evaluate_agent(self, batch_size=None):
        """Greedy-Q rollouts of `test_episodes` episodes on random test environments (reference dqn.py:514-602).
        Returns (mean score, mean solution) for TestMetric.BEST / FINAL.

        The reference fills `batch_size` (default: the minibatch size) slots, steps them together -- so `norm.max()`
        (mpnn.py:102) is the largest degree among the graphs of that group -- and refills when the group is done; per
        episode it draws, in order, the environment (`random.sample`), the graph (`gg.get()`) and the spins
        (`np.random.randint`).  Same draws, same groups here; every group is one device rollout."""
        k = self.test_episodes
        bsz = self.minibatch_size if batch_size is None else int(batch_size)
        graphs, spins = [], []
        for _ in range(k):
            e = random.sample(self.test_envs, k=1)[0]                        # get_random_env, dqn.py:242-248
            graphs.append(np.asarray(e.gg.get()))                            # env.reset(): spinsystem.py:188-198
            spins.append(2 * np.random.randint(2, size=self.n_spins) - 1)    # spinsystem.py:294
        t_env = self.test_envs[0]
        gs = engine.GraphSet(np.stack(graphs), device=self.device,
                             min_cut=t_env.optimisation_target == OptimisationTarget.MIN_CUT)
        deg = gs.gstat[:, 0].cpu().numpy()
        w = self.network.engine_weights(self.device)
        scores, sols = np.zeros(k), np.zeros(k)
        for g0 in range(0, k, bsz):
            g1 = min(k, g0 + bsz)
            env = engine.BatchedSpinSystem(gs, g1 - g0, t_env.max_steps, t_env.basin_reward)
            env.reset(spins=np.stack(spins[g0:g1]), graph_idx=np.arange(g0, g1, dtype=np.int32))
            env.rollout(w, norm_max=float(max(1, deg[g0:g1].max())))
            ep = env.episodes()
            if self.test_metric == TestMetric.BEST:
                scores[g0:g1], sols[g0:g1] = ep["best_score"], ep["best_cut"]
            else:
                scores[g0:g1], sols[g0:g1] = ep["score"], ep["cut"]
        self.last_test_scores, self.last_test_solutions = scores, sols
        return (np.mean(scores), np.mean(sols))

    def save(self, path='network.pth'):
        if os.path.dirname(path):
            os.makedirs(os.path.dirname(path), exist_ok=True)
        torch.save(self.network.state_dict(), path)

    def load(self, path):
        self.network.load_state_dict(torch.load(path, map_location=self.device))
