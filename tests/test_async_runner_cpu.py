"""Host logic of the asynchronous runner (rlpyt_b200/runners/async_rl.py; reference rlpyt/runners/async_rl.py:21-612):
thread roles, double-buffer hand-shake, throttle arithmetic, logging rows, shutdown and error paths - with stand-in
sampler / algorithm / replay objects (no GPU here; the GPU test runs the real classes)."""
import threading
import time

import numpy as np
import pytest
import torch

from rlpyt_b200.agents.base import BaseAgent
from rlpyt_b200.runners.async_rl import AsyncRl, AsyncRlEval
from rlpyt_b200.samplers.collections import BatchSpec
from rlpyt_b200.utils.logging import TabularLogger
from rlpyt_b200.utils.synchronize import RWLock


class FakeReplay:
    def __init__(self):
        self.appended = []
        self.lock = threading.Lock()

    def append_samples(self, samples):
        with self.lock:
            self.appended.append(int(samples["itr"]))


class FakeSampler:
    """Publishes {'itr': itr} into double_buffer[db_idx]; checks that a buffer is never overwritten before it was consumed."""
    mid_batch_reset = True

    def __init__(self, T=4, B=8, step_s=0.002, fail_at=None, eval_trajs=2):
        self.batch_spec = BatchSpec(T, B)
        self.step_s, self.fail_at, self.eval_trajs = step_s, fail_at, eval_trajs
        self.double_buffer = ({"itr": -1, "fresh": False}, {"itr": -1, "fresh": False})
        self.calls, self.shutdowns, self.initialized = [], 0, False
        self.device = None

    @property
    def batch_size(self):
        return self.batch_spec.size

    def async_initialize(self, agent, bootstrap_value=False, traj_info_kwargs=None, seed=None, device=None):
        # ``device``: the runner passes its CUDA device where one exists; this stand-in stays on the host (self.device None)
        self.agent = agent
        self.traj_info_kwargs = traj_info_kwargs
        return self.double_buffer, dict(observation=np.zeros(3))

    def initialize(self, affinity):
        self.initialized = True
        self.affinity = affinity

    def obtain_samples(self, itr, db_idx):
        if self.fail_at is not None and itr == self.fail_at:
            raise ValueError("env exploded")
        time.sleep(self.step_s)
        buf = self.double_buffer[db_idx]
        assert not buf["fresh"], "buffer overwritten before the copier consumed it"
        buf["itr"], buf["fresh"] = itr, True
        self.calls.append((itr, db_idx))
        return [dict(Length=10, Return=float(itr))] if itr % 2 == 0 else []

    def evaluate_agent(self, itr):
        return [dict(Length=7, Return=1.0) for _ in range(self.eval_trajs)]

    def acquire_batch(self, db_idx, stream=None):
        return self.double_buffer[db_idx]

    def release_batch(self, db_idx, stream=None):
        self.double_buffer[db_idx]["fresh"] = False

    def shutdown(self):
        self.shutdowns += 1


class FakeAlgo:
    opt_info_fields = ("loss",)
    bootstrap_value = False
    discount = 0.9

    def __init__(self, batch_size=16, replay_ratio=2, updates_per_sync=1, min_steps_learn=64, opt_s=0.0):
        self.batch_size, self.replay_ratio = batch_size, replay_ratio
        self.updates_per_optimize = updates_per_sync
        self.min_steps_learn, self.opt_s = min_steps_learn, opt_s
        self.update_counter = 0
        self.calls = []
        self.replay = FakeReplay()

    def async_initialize(self, agent, sampler_n_itr, batch_spec, mid_batch_reset, examples, world_size=1):
        self.n_itr = sampler_n_itr
        assert examples is not None
        return self.replay

    def optim_initialize(self, rank=0):
        self.rank = rank

    def samples_to_buffer(self, samples):
        return samples

    def optimize_agent(self, itr, samples=None, sampler_itr=None):
        assert samples is None
        time.sleep(self.opt_s)
        self.calls.append((itr, sampler_itr, len(self.replay.appended)))
        self.update_counter += self.updates_per_optimize
        from collections import namedtuple
        return namedtuple("OptInfo", ["loss"])(loss=[float(itr)])

    def optim_state_dict(self):
        return {}


class FakeAgent:
    def __init__(self):
        self.sent, self.device_idx = 0, "unset"

    def to_device(self, cuda_idx=None):
        self.device_idx = cuda_idx

    def send_shared_memory(self):
        self.sent += 1

    def state_dict(self):
        return {}


def _runner(cls=AsyncRl, sampler=None, algo=None, n_steps=32 * 40, log_interval_steps=32 * 10, **kw):
    sampler = sampler or FakeSampler()
    algo = algo or FakeAlgo()
    agent = FakeAgent()
    logger = TabularLogger(quiet=True)
    r = cls(algo=algo, agent=agent, sampler=sampler, n_steps=n_steps, affinity=dict(cuda_idx=None), seed=1,
            log_interval_steps=log_interval_steps, logger=logger, **kw)
    r.throttle_wait = 0.002
    return r, sampler, algo, agent, logger


def test_async_rl_runs_all_sampler_iterations_and_throttles_the_optimizer():
    r, sampler, algo, agent, logger = _runner()
    n_opt = r.train()
    n_itr = 40
    assert r.n_itr == n_itr and [c[0] for c in sampler.calls] == list(range(n_itr))
    assert [c[1] for c in sampler.calls] == [i % 2 for i in range(n_itr)]                 # double buffer toggles
    assert algo.replay.appended == list(range(n_itr))                                     # every batch, once, in order
    assert sampler.initialized and sampler.shutdowns == 1
    assert sampler.traj_info_kwargs == dict(discount=0.9)
    # throttle (async_rl.py:172-176): optimizer iteration k may start only when sampler_itr >= 1 + min_steps//bs + k*delta
    bs = sampler.batch_size
    delta = algo.batch_size * 1 * algo.updates_per_optimize / (bs * algo.replay_ratio)
    first = 1 + algo.min_steps_learn // bs
    assert n_opt == len(algo.calls) > 0
    for k, (itr, sampler_itr, n_appended) in enumerate(algo.calls):
        assert itr == k and sampler_itr >= first + k * delta - 1e-9
    # the optimizer cannot run ahead: the replay-ratio bound on the number of iterations it may have done
    assert len(algo.calls) <= (n_itr - first) / delta + 1
    assert agent.sent == len(algo.calls)                                                  # parameters sent after every optimize_agent
    # logging: one table per log interval (+ final), with the reference's rows
    t = logger.tables[-1]
    for key in ("Diagnostics/SamplerIteration", "Diagnostics/CumSteps", "Diagnostics/CumUpdates", "Diagnostics/ReplayRatio",
                "Diagnostics/StepsPerSecond", "Diagnostics/UpdatesPerSecond", "Diagnostics/OptThrottle",
                "Diagnostics/CumCompletedTrajs", "lossAverage", "ReturnAverage"):
        assert key in t, key
    assert t["Diagnostics/CumSteps"] == (n_itr - 1) * bs and t["Diagnostics/CumUpdates"] == algo.update_counter
    assert t["Diagnostics/CumCompletedTrajs"] == n_itr // 2
    assert len(logger.tables) >= 3 and logger.snapshots


def test_async_rl_slow_optimizer_never_blocks_the_sampler_beyond_the_double_buffer():
    algo = FakeAlgo(opt_s=0.01, min_steps_learn=0)
    r, sampler, algo, agent, logger = _runner(algo=algo, sampler=FakeSampler(step_s=0.0005), n_steps=32 * 30)
    r.train()
    assert algo.replay.appended == list(range(30))            # the copier, not the optimizer, frees the buffers
    assert 0 < len(algo.calls) < 30                           # the optimizer did fewer iterations than its bound allowed


def test_async_rl_eval_variant_logs_offline_evaluations():
    r, sampler, algo, agent, logger = _runner(cls=AsyncRlEval)
    r.train()
    assert [c[0] for c in sampler.calls] == list(range(41))   # n_itr + 1: the last evaluation (async_rl.py:546)
    t = logger.tables[0]
    assert t["Diagnostics/StepsInEval"] == 14 and t["Diagnostics/TrajsInEval"] == 2      # the eval before any optimization
    assert "Diagnostics/CumEvalTime" in logger.tables[-1] and "Diagnostics/NonEvalSamplesPerSecond" in logger.tables[-1]


def test_async_rl_sampler_failure_surfaces_in_train_and_everything_is_joined():
    r, sampler, algo, agent, logger = _runner(sampler=FakeSampler(fail_at=5))
    with pytest.raises(RuntimeError, match="sampler thread failed") as e:
        r.train()
    assert isinstance(e.value.__cause__, ValueError)
    assert not r.sampler_thread.is_alive() and not r.memcpy_thread.is_alive()
    assert algo.replay.appended == list(range(5))


def test_async_rl_affinity_structures():
    from rlpyt_b200.utils.collections import AttrDict
    r, *_ = _runner()
    r.affinity = AttrDict(sampler=dict(workers_cpus=[1, 2]), optimizer=[dict(cuda_idx=3, cpus=[0])])
    a = r._affinities()
    assert a.sampler == dict(workers_cpus=[1, 2]) and a.optimizer == dict(cuda_idx=3, cpus=[0])
    r.affinity = dict(cuda_idx=0, workers_cpus=[4])
    a = r._affinities()
    assert a.sampler == a.optimizer == dict(cuda_idx=0, workers_cpus=[4])


def test_rwlock_readers_share_writers_exclude():
    lock = RWLock()
    state = dict(readers=0, max_readers=0, writer_saw_readers=False)
    gate = threading.Barrier(3)

    def reader():
        gate.wait()
        with lock:
            state["readers"] += 1
            state["max_readers"] = max(state["max_readers"], state["readers"])
            time.sleep(0.05)
            state["readers"] -= 1

    def writer():
        gate.wait()
        time.sleep(0.01)
        with lock.write_lock:
            state["writer_saw_readers"] = state["readers"] != 0

    ts = [threading.Thread(target=f) for f in (reader, reader, writer)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert state["max_readers"] == 2 and not state["writer_saw_readers"]


class _LinearAgent(BaseAgent):
    def __init__(self):
        super().__init__(ModelCls=lambda: torch.nn.Linear(3, 2))

    def initialize(self):
        self.model = self.ModelCls()


def test_agent_parameter_channel_staging_semantics():
    """agents/base.py:218-243: the sampler's copy changes only at recv, to the LAST sent parameters; the optimizer's
    parameters are never written by the channel."""
    a = _LinearAgent()
    a.initialize()
    twin = a.async_twin()
    w0 = a.model.weight.detach().clone()
    assert twin.model is not a.model and torch.equal(twin.model.weight, w0)
    with torch.no_grad():
        a.model.weight.add_(1.0)
    twin.recv_shared_memory()
    assert torch.equal(twin.model.weight, w0)                 # nothing was sent yet
    a.send_shared_memory()
    with torch.no_grad():
        a.model.weight.add_(1.0)                              # the optimizer keeps stepping after the send
    assert torch.equal(twin.model.weight, w0)                 # ... and the sampler is still mid-batch on the old set
    twin.recv_shared_memory()
    assert torch.equal(twin.model.weight, w0 + 1.0)           # the sent snapshot, not the live parameters
    twin.recv_shared_memory()
    assert torch.equal(twin.model.weight, w0 + 1.0) and torch.equal(a.model.weight, w0 + 2.0)
    a.recv_shared_memory()
    twin.send_shared_memory()                                 # wrong-side calls are no-ops
    assert torch.equal(a.model.weight, w0 + 2.0)
