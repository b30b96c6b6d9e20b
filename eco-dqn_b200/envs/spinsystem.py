"""Single-environment facade with the reference's SpinSystem surface, backed by the batched device engine (B = 1).

Mirrors reference src/envs/spinsystem.py: SpinSystemFactory.get (:29-48) and the parts of SpinSystemBase that
callers touch (:132-177 attributes, reset :183-259, step :355-559, get_observation :561-574,
get_allowed_action_states :576-593).  Only the Max-Cut ECO-DQN configuration is accelerated; anything else raises
NotImplementedError at construction (SURVEY.md section 8b) -- there is no silent fallback.

This class exists for API compatibility (solvers, user scripts).  Throughput comes from
eco_dqn_b200.engine.BatchedSpinSystem / experiments.utils.test_network, which step thousands of episodes per launch.
"""
import copy

import numpy as np
import torch

from .. import engine
from .utils import (DEFAULT_OBSERVABLES, EdgeType, ExtraAction, GraphGenerator, Observable, OptimisationTarget,
                    RandomErdosRenyiGraphGenerator, RewardSignal, SpinBasis, Stopping, calculate_cut,
                    calculate_cut_changes)


class MaxCutScorer:
    """Host-side view of MaximumCutUnbiasedScorer (reference src/envs/score_solver.py:343-419) for callers that
    query the scorer directly (solver.py:66,113; experiments/utils.py:159,190)."""

    def __init__(self):
        self._max_local_reward = 1
        self._solution_quality_normalizer = 1
        self._invalidity_normalizer = 1
        self._lower_bound = 0

    def set_constants(self, mlr, qn, lb):
        self._max_local_reward, self._solution_quality_normalizer, self._lower_bound = mlr, qn, lb

    def get_solution(self, spins, matrix):
        return calculate_cut(spins, matrix)

    def get_solution_quality(self, spins, matrix):
        return self.get_solution(spins, matrix) + abs(min(0, self._lower_bound))

    def get_score(self, spins, matrix):
        return self.get_solution_quality(spins, matrix)

    def get_normalized_score(self, spins, matrix):
        return self.get_solution_quality(spins, matrix) / self._solution_quality_normalizer

    def get_score_mask(self, spins, matrix):
        return calculate_cut_changes(spins, matrix)

    get_solution_quality_mask = get_score_mask

    def get_normalized_score_mask(self, spins, matrix):
        return self.get_score_mask(spins, matrix) / self._solution_quality_normalizer

    def get_invalidity_degree(self, spins, matrix):
        return 0

    def is_valid(self, spins, matrix):
        return True


class MinCutScorer(MaxCutScorer):
    """Host-side view of MinimumCutUnbiasedSolver (reference src/envs/score_solver.py:423-505): every mask is the negated
    cut change, the quality is normaliser - cut."""

    def get_solution_quality(self, spins, matrix):
        return max(0, self._solution_quality_normalizer) - self.get_solution(spins, matrix)     # :219-222

    def get_score_mask(self, spins, matrix):
        return -calculate_cut_changes(spins, matrix)

    get_solution_quality_mask = get_score_mask

    def get_normalized_score_mask(self, spins, matrix):
        return self.get_score_mask(spins, matrix) / self._solution_quality_normalizer


class _ActionSpace:
    def __init__(self, n_actions):
        self.n = n_actions
        self.actions = np.arange(self.n)

    def sample(self, n=1):
        return np.random.choice(self.actions, n)


class _ObservationSpace:
    def __init__(self, n_spins, n_observables):
        self.shape = [n_spins, n_observables]


class SpinSystemFactory(object):
    @staticmethod
    def get(graph_generator=None, max_steps=20, observables=DEFAULT_OBSERVABLES, reward_signal=RewardSignal.DENSE,
            extra_action=ExtraAction.PASS, optimisation_target=OptimisationTarget.ENERGY, spin_basis=SpinBasis.SIGNED,
            norm_rewards=False, memory_length=None, horizon_length=None, stag_punishment=None, basin_reward=None,
            reversible_spins=True, init_snap=None, seed=None, stopping=Stopping.NORMAL):
        return SpinSystemBase(graph_generator, max_steps, observables, reward_signal, extra_action, optimisation_target,
                              spin_basis, norm_rewards, memory_length, horizon_length, stag_punishment, basin_reward,
                              reversible_spins, init_snap, seed, stopping)


def check_supported(observables, reward_signal, extra_action, optimisation_target, spin_basis, norm_rewards,
                    memory_length, horizon_length, stag_punishment, reversible_spins, init_snap, stopping, max_steps):
    """The accelerated configurations: ECO-DQN as every reference script uses it (SURVEY.md appendix A), and S2V-DQN as
    experiments/pretrained_agent/test_s2v.py configures it (observables=[SPIN_STATE], RewardSignal.DENSE, irreversible
    spins, no basin reward) -- with SpinBasis.SIGNED, because BINARY is broken in the reference's own drivers."""
    assert observables[0] == Observable.SPIN_STATE, "First observable must be Observation.SPIN_STATE."
    problems = []
    s2v = not reversible_spins
    if s2v:
        if list(observables) != [Observable.SPIN_STATE]:
            problems.append("irreversible spins (S2V-DQN): observables must be [Observable.SPIN_STATE]")
        if reward_signal != RewardSignal.DENSE:
            problems.append("irreversible spins (S2V-DQN): reward_signal must be RewardSignal.DENSE")
    else:
        if list(observables) != DEFAULT_OBSERVABLES:
            problems.append("observables must be DEFAULT_OBSERVABLES")
        if reward_signal != RewardSignal.BLS:
            problems.append("reward_signal must be RewardSignal.BLS")
    if optimisation_target not in (OptimisationTarget.CUT, OptimisationTarget.MIN_CUT):
        problems.append("optimisation_target must be OptimisationTarget.CUT or MIN_CUT (got %s)" % optimisation_target)
    if not norm_rewards:
        problems.append("norm_rewards must be True")
    if extra_action != ExtraAction.NONE:
        problems.append("extra_action must be ExtraAction.NONE")
    if spin_basis != SpinBasis.SIGNED:
        problems.append("spin_basis must be SpinBasis.SIGNED (BINARY is broken in the reference's own drivers)")
    if memory_length is not None:
        problems.append("memory_length must be None (infinite memory)")
    if horizon_length is not None and horizon_length != max_steps:
        problems.append("horizon_length must be None or max_steps")
    if stag_punishment is not None:
        problems.append("stag_punishment must be None")
    if init_snap is not None:
        problems.append("init_snap is not supported (it is broken in the reference as well)")
    if stopping != Stopping.NORMAL:
        problems.append("stopping must be Stopping.NORMAL")
    if problems:
        raise NotImplementedError("configuration outside the accelerated Max-Cut ECO-DQN / S2V-DQN paths: " + "; ".join(problems))


class SpinSystemBase:
    def __init__(self, graph_generator=None, max_steps=20, observables=DEFAULT_OBSERVABLES,
                 reward_signal=RewardSignal.DENSE, extra_action=ExtraAction.PASS,
                 optimisation_target=OptimisationTarget.ENERGY, spin_basis=SpinBasis.SIGNED, norm_rewards=False,
                 memory_length=None, horizon_length=None, stag_punishment=None, basin_reward=None,
                 reversible_spins=False, init_snap=None, seed=None, stopping=Stopping.NORMAL, device=None):
        check_supported(observables, reward_signal, extra_action, optimisation_target, spin_basis, norm_rewards,
                        memory_length, horizon_length, stag_punishment, reversible_spins, init_snap, stopping, max_steps)
        if not reversible_spins and basin_reward is not None:
            raise NotImplementedError("irreversible spins (S2V-DQN): basin_reward must be None")
        if seed is not None:
            np.random.seed(seed)
        self.observables = list(enumerate(observables))
        self.extra_action = extra_action
        if graph_generator is not None:
            assert isinstance(graph_generator, GraphGenerator), "graph_generator must be a GraphGenerator implementation."
            self.gg = graph_generator
        else:
            self.gg = RandomErdosRenyiGraphGenerator(n_spins=20, p_connection=0.15, edge_type=EdgeType.DISCRETE)
        if self.gg.biased:
            raise NotImplementedError("biased graphs are outside the accelerated path")
        self.n_spins = self.gg.n_spins
        self.max_steps = max_steps
        self.reward_signal = reward_signal
        self.norm_rewards = norm_rewards
        self.n_actions = self.n_spins
        self.action_space = _ActionSpace(self.n_actions)
        self.observation_space = _ObservationSpace(self.n_spins, len(self.observables))
        self.stopping_type = stopping
        self.optimisation_target = optimisation_target
        self.scorer = MinCutScorer() if optimisation_target == OptimisationTarget.MIN_CUT else MaxCutScorer()
        self.spin_basis = spin_basis
        self.memory_length = memory_length
        self.horizon_length = horizon_length if horizon_length is not None else self.max_steps
        self.stag_punishment = stag_punishment
        self.basin_reward = basin_reward
        self.reversible_spins = reversible_spins
        self.bias = None
        self._device = device
        self._graphset = None
        self._graph_key = None
        self._env = None
        self._ep = None
        self.matrix = None
        self.reset()

    # ------------------------------------------------------------------ device plumbing
    def _bind_graph(self, matrix):
        key = (id(matrix), matrix.shape)
        if self._graphset is None or key != self._graph_key:
            # integer couplings in [-127, 127]: the int8 path; anything else (EdgeType.RANDOM): the fp64 weighted path
            self._graphset = engine.graph_set(np.asarray(matrix)[None], device=self._device,
                                              min_cut=self.optimisation_target == OptimisationTarget.MIN_CUT)
            self._graph_key = key
            self._env = self._new_env()
            sc = self._graphset.gscal.cpu().numpy()[0]
            self.scorer.set_constants(sc[0], sc[1], sc[2])
        self.matrix = matrix
        self.matrix_obs = matrix

    def _new_env(self):
        return engine.BatchedSpinSystem(self._graphset, 1, self.max_steps, self.basin_reward,
                                        reversible_spins=self.reversible_spins,
                                        dense_reward=self.reward_signal == RewardSignal.DENSE)

    def _episode(self):
        if self._ep is None:
            self._ep = self._env.episodes()[0]
        return self._ep

    # ------------------------------------------------------------------ reference surface
    def reset(self, spins=None):
        self._bind_graph(self.gg.get())
        n = self.n_spins
        if spins is None:
            if self.reversible_spins:
                spins = 2 * np.random.randint(2, size=n) - 1      # spinsystem.py:294
            else:
                spins = -np.ones(n, dtype=np.int64)               # spinsystem.py:296-297
        else:
            spins = np.asarray(spins)
            if not np.isin(spins, [-1, 1]).all():                 # spinsystem.py:604-606
                raise Exception("SpinSystem is configured for signed spins ([-1,1]).")
        self._env.reset(spins=np.asarray(spins).reshape(1, n))
        self._ep = None
        return self.get_observation()

    def seed(self, seed):
        return self.seed

    def set_seed(self, seed):
        self.seed = seed
        np.random.seed(seed)

    def step(self, action):
        if self._env.current_step + 1 > self.max_steps:
            print("The environment has already returned done. Stop it!")
            raise NotImplementedError
        rew, done = self._env.step(torch.tensor([int(action)], dtype=torch.int32))
        self._ep = None
        ep = self._episode()
        return (self.get_observation(), float(ep["last_reward"]), bool(ep["flags"] & 1), None)

    def get_observation(self):
        rows = self._env.observation()[0].double().cpu().numpy()
        return np.vstack((rows[:len(self.observables)], self.matrix_obs))     # S2V-DQN: the spin row only

    def get_allowed_action_states(self):
        return (-1, 1) if self.reversible_spins else -1                       # spinsystem.py:576-594 (SIGNED)

    # ------------------------------------------------------------------ attributes callers read
    @property
    def state(self):
        return self._env.observation()[0].double().cpu().numpy()[:len(self.observables)]

    @property
    def current_step(self):
        return int(self._episode()["step"])

    @property
    def score(self):
        return float(self._episode()["score"])

    @property
    def normalized_score(self):
        return float(self._episode()["nscore"])

    @property
    def best_score(self):
        return float(self._episode()["best_score"])

    @property
    def best_score_normalized(self):
        return float(self._episode()["best_nscore"])

    @property
    def best_obs_score(self):
        return self.best_score

    @property
    def best_solution(self):
        return float(self._episode()["best_cut"])

    @property
    def best_spins(self):
        return self._env.results()[1][0].double().cpu().numpy()

    @property
    def best_obs_spins(self):
        return self.best_spins

    def __deepcopy__(self, memo):
        new = self.__class__.__new__(self.__class__)
        for k, v in self.__dict__.items():
            if k in ("_graphset", "_env", "_ep", "matrix", "matrix_obs", "gg"):
                continue
            setattr(new, k, copy.deepcopy(v, memo))
        new.gg = self.gg                      # generators are shared like the graphs they hold
        new._graphset, new._graph_key = self._graphset, self._graph_key
        new.matrix, new.matrix_obs = self.matrix, self.matrix_obs
        new._env = new._new_env()
        new._env._ws.copy_(self._env._ws)
        new._env.current_step = self._env.current_step
        new._env._is_reset = self._env._is_reset
        new._ep = None
        return new
