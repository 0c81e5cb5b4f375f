"""The UNMODIFIED reference (astooke/rlpyt, copied into oracle/_ref by oracle/reference_install.py)
driven through its own public API for bench.py's ``--impl reference`` arm:

    GpuSampler(EnvCls, batch_T, batch_B).initialize(agent, affinity, seed, bootstrap_value)
    loop: agent.sample_mode -> sampler.obtain_samples -> agent.train_mode -> algo.optimize_agent
    (the body of rlpyt/runners/minibatch_rl.py:246-263 without logging)

with ``affinity = dict(cuda_idx=None, workers_cpus=[...])`` = the reference's pure-CPU path (batched action
serving in the master on torch-CPU, env stepping in forked worker processes) or ``cuda_idx=0`` = stock
PyTorch kernels on the B200 (context leg).  None of this repo's kernels, models or samplers are on that
path; the only thing supplied is the synthetic Atari-shaped environment (``atari_py`` is not installed and
there is no network), written against the reference's ``Env`` interface with the same behaviour as
rlpyt_b200/envs/synthetic.py.
"""
import sys
import time
from collections import namedtuple

import numpy as np

from oracle.reference_install import DEST as REF, available  # noqa: F401

EnvInfo = namedtuple("EnvInfo", ["game_score", "traj_done"])     # module level: the reference pickles an example


def _import():
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import torch  # noqa: F401
    from rlpyt.envs.base import Env, EnvStep
    from rlpyt.spaces.int_box import IntBox
    return Env, EnvStep, IntBox


def make_env_cls():
    Env, EnvStep, IntBox = _import()
    class SyntheticAtariEnv(Env):
        """Same dynamics and per-step cost as rlpyt_b200.envs.synthetic.SyntheticAtariEnv."""

        _POOLS = {}

        def __init__(self, image_shape=(4, 84, 84), n_actions=6, p_done=1 / 500., p_reward=0.04, pool_frames=32, seed=0):
            self.image_shape = tuple(image_shape)
            self._action_space = IntBox(low=0, high=n_actions)
            self._observation_space = IntBox(low=0, high=256, shape=self.image_shape, dtype="uint8")
            key = (self.image_shape, pool_frames)
            if key not in SyntheticAtariEnv._POOLS:
                rng = np.random.default_rng(1234)
                SyntheticAtariEnv._POOLS[key] = rng.integers(0, 256, size=(pool_frames,) + self.image_shape, dtype=np.uint8)
            self._pool = SyntheticAtariEnv._POOLS[key]
            self.p_done, self.p_reward = p_done, p_reward
            self.seed(seed)

        def seed(self, seed):
            self._rng = np.random.default_rng(seed)
            self._cursor = int(self._rng.integers(0, len(self._pool)))

        def reset(self):
            self._cursor = int(self._rng.integers(0, len(self._pool)))
            return self._pool[self._cursor]

        def step(self, action):
            u = self._rng.random(2)
            self._cursor = (self._cursor + 1 + int(action)) % len(self._pool)
            reward = 0.0
            if u[0] < self.p_reward:
                reward = 1.0 if u[0] < self.p_reward / 2 else -1.0
            done = bool(u[1] < self.p_done)
            return EnvStep(self._pool[self._cursor], np.float32(reward), done, EnvInfo(int(reward), done))

        @property
        def horizon(self):
            return 27000

    return SyntheticAtariEnv


class ReferenceLoop:
    """sampler + agent + algo of the reference, built the way rlpyt/runners/minibatch_rl.py:74-96 builds them."""

    def __init__(self, batch_T, batch_B, env_kwargs, ppo_kwargs, workers_cpus, cuda_idx=None, seed=0, n_itr=10 ** 6):
        _import()
        import torch
        from rlpyt.agents.pg.atari import AtariFfAgent
        from rlpyt.algos.pg.ppo import PPO
        from rlpyt.samplers.parallel.gpu.sampler import GpuSampler
        from rlpyt.utils.seed import set_seed
        set_seed(seed)
        self.torch = torch
        self.cuda_idx = cuda_idx
        self.sampler = GpuSampler(EnvCls=make_env_cls(), env_kwargs=env_kwargs, batch_T=batch_T, batch_B=batch_B,
                                  max_decorrelation_steps=20)
        self.agent = AtariFfAgent()
        self.algo = PPO(**ppo_kwargs)
        affinity = dict(cuda_idx=cuda_idx, workers_cpus=list(workers_cpus), set_affinity=True)
        examples = self.sampler.initialize(agent=self.agent, affinity=affinity, seed=seed + 1, bootstrap_value=True,
                                           traj_info_kwargs=dict(discount=ppo_kwargs.get("discount", 0.99)))
        self.agent.to_device(cuda_idx)                          # minibatch_rl.py:84
        self.algo.initialize(agent=self.agent, n_itr=n_itr, batch_spec=self.sampler.batch_spec,
                             mid_batch_reset=self.sampler.mid_batch_reset, examples=examples)
        self.itr = 0
        self.t_sample = 0.0
        self.t_optimize = 0.0

    def _sync(self):
        if self.cuda_idx is not None:
            self.torch.cuda.synchronize()

    def step(self):
        """One iteration of minibatch_rl.py:255-260."""
        t0 = time.perf_counter()
        self.agent.sample_mode(self.itr)
        samples, traj_infos = self.sampler.obtain_samples(self.itr)
        t1 = time.perf_counter()
        self.agent.train_mode(self.itr)
        info = self.algo.optimize_agent(self.itr, samples)
        self._sync()
        t2 = time.perf_counter()
        self.t_sample += t1 - t0
        self.t_optimize += t2 - t1
        self.itr += 1
        return info

    def reset_timers(self):
        self.t_sample = self.t_optimize = 0.0

    def shutdown(self):
        self.sampler.shutdown()
