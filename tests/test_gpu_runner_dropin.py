"""Drop-in proof (north_star: "existing runners ... drop in"): the UNMODIFIED reference runner
``rlpyt.runners.minibatch_rl.MinibatchRl`` (from oracle/_ref, see oracle/reference_install.py) drives
this repo's GpuSampler / AlternatingSampler + AtariFfAgent + PPO (and SerialSampler + A2C, BASELINE.json configs[0]
plumbing) through its own ``startup()`` / ``train()``: sampler.initialize(agent, affinity, seed, bootstrap_value,
traj_info_kwargs, rank, world_size) -> agent.to_device -> algo.initialize(agent, n_itr, batch_spec, mid_batch_reset,
examples, world_size, rank) -> [sample_mode, obtain_samples, train_mode, optimize_agent, store/log diagnostics] x n
-> shutdown (rlpyt/runners/minibatch_rl.py:52-96, 246-263).  Only ``pyprind`` (a progress bar the image does not
have) is stubbed."""
import sys
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _reference_runner():
    from oracle import reference_install
    if not reference_install.available():
        pytest.skip("the reference package is not available (oracle/_ref was not built)")
    if reference_install.DEST not in sys.path:
        sys.path.insert(0, reference_install.DEST)
    if "pyprind" not in sys.modules:                      # rlpyt/utils/prog_bar.py:3
        stub = types.ModuleType("pyprind")

        class ProgBar:
            def __init__(self, *a, **k):
                self.active = True

            def update(self, *a, **k):
                pass

            def stop(self):
                self.active = False
        stub.ProgBar = ProgBar
        sys.modules["pyprind"] = stub
    from rlpyt.runners.minibatch_rl import MinibatchRl
    return MinibatchRl


@pytest.mark.parametrize("kind", ["gpu_ppo", "alternating_ppo", "serial_a2c"])
def test_reference_minibatch_rl_drives_b200_classes(kind, capsys):
    MinibatchRl = _reference_runner()
    from rlpyt_b200.agents.pg.atari import AtariFfAgent
    from rlpyt_b200.algos.pg.a2c import A2C
    from rlpyt_b200.algos.pg.ppo import PPO
    from rlpyt_b200.envs.synthetic import SyntheticAtariEnv
    from rlpyt_b200.samplers.parallel.gpu.alternating_sampler import AlternatingSampler
    from rlpyt_b200.samplers.parallel.gpu.sampler import GpuSampler
    from rlpyt_b200.samplers.serial.sampler import SerialSampler
    env_kwargs = dict(image_shape=(4, 36, 36), n_actions=5, p_done=0.05, p_reward=0.3)
    T, B = (5, 8) if kind == "serial_a2c" else (8, 8)
    cls = dict(gpu_ppo=GpuSampler, alternating_ppo=AlternatingSampler, serial_a2c=SerialSampler)[kind]
    sampler = cls(EnvCls=SyntheticAtariEnv, env_kwargs=env_kwargs, batch_T=T, batch_B=B, max_decorrelation_steps=3)
    algo = A2C() if kind == "serial_a2c" else PPO(minibatches=2, epochs=2)
    agent = AtariFfAgent()
    affinity = dict(cuda_idx=0, workers_cpus=[None, None], set_affinity=False)
    n_itr_want = 6
    runner = MinibatchRl(algo=algo, agent=agent, sampler=sampler, n_steps=n_itr_want * T * B, seed=3, affinity=affinity,
                         log_interval_steps=2 * T * B)
    w0 = None
    orig_startup = runner.startup

    def startup():
        n = orig_startup()
        nonlocal w0
        w0 = {k: v.detach().clone() for k, v in agent.state_dict().items()}
        return n
    runner.startup = startup
    runner.train()                                        # the reference's own loop, start to shutdown
    assert runner.n_itr == n_itr_want and algo.update_counter == n_itr_want * (1 if kind == "serial_a2c" else 4)
    out = capsys.readouterr().out
    assert "StepsPerSecond" in out and "CumUpdates" in out and "gradNorm" in out       # the reference's logger table
    snap = runner.get_itr_snapshot(n_itr_want - 1)
    assert snap["cum_steps"] == (n_itr_want - 1) * T * B and "optimizer_state_dict" in snap
    moved = [float((v - w0[k]).abs().max()) for k, v in agent.state_dict().items()]
    assert max(moved) > 0 and all(np.isfinite(moved))     # the agent the runner holds was trained
    assert all(p.is_cuda for p in agent.parameters())
