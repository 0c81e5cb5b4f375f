#!/usr/bin/env python
"""Generate golden fixtures by CALLING the unmodified reference (never copying it).

Run in the build container only (the GPU box has no /root/reference):

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py [--only returns,loss,...]

Writes tests/golden/<group>.npz (compressed).  Each group stores the exact inputs and
the reference's outputs, so the tests never need the reference at run time.
"""
import argparse
import os
import sys
import types

import numpy as np

REF = os.environ.get("RLPYT_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))


def _import_reference():
    sys.dont_write_bytecode = True
    if REF not in sys.path:
        sys.path.insert(0, REF)
    # rlpyt.utils.prog_bar needs pyprind (absent, no network): 6-line stub.
    if "pyprind" not in sys.modules:
        stub = types.ModuleType("pyprind")

        class ProgBar:  # noqa: D401 - stub
            def __init__(self, *a, **k):
                self.active = True

            def update(self, *a, **k):
                pass

            def stop(self):
                self.active = False
        stub.ProgBar = ProgBar
        sys.modules["pyprind"] = stub


def _save(name, arrays):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"wrote {path}: {len(arrays)} arrays, {os.path.getsize(path)/1024:.1f} KiB")


# --------------------------------------------------------------------------- returns
def returns_inputs(seed, T, B, p_done=0.01, sparse=False, pattern=None):
    """Synthetic inputs of SURVEY.md section 8(d) row 2."""
    rng = np.random.default_rng(seed)
    if sparse:
        reward = rng.choice(np.array([-1, 0, 1], dtype=np.float32), size=(T, B),
                            p=[0.02, 0.96, 0.02]).astype(np.float32)
    else:
        reward = rng.standard_normal((T, B), dtype=np.float32)
    value = rng.standard_normal((T, B), dtype=np.float32)
    done = rng.random((T, B)) < p_done
    bv = rng.standard_normal((1, B), dtype=np.float32)
    if pattern == "edges":  # done at t=0, t=T-1, an all-done column, a never-done column
        done[:] = False
        done[0, 0] = True
        done[T - 1, 1 % B] = True
        done[:, 2 % B] = True
        if B > 3:
            done[T // 2, 3] = True
            done[T // 2 + 1 if T // 2 + 1 < T else T - 1, 3] = True
    return reward, value, done, bv


RETURNS_CASES = [
    # name, seed, T, B, p_done, sparse, pattern
    ("kat", None, 4, 2, None, False, None),
    ("t1", 11, 1, 3, 0.3, False, None),
    ("t2b1", 12, 2, 1, 0.3, False, None),
    ("cfg1", 13, 5, 8, 0.1, False, None),
    ("edges", 14, 16, 7, 0.0, False, "edges"),
    ("ragged", 15, 37, 61, 0.05, False, None),
    ("sparse", 16, 64, 40, 0.01, True, None),
    ("cfg2", 0, 128, 256, 0.01, False, None),
]
GAMMAS_LAMBDAS = [(0.99, 1.0), (0.99, 0.98), (0.99, 0.95), (1.0, 0.9), (0.9, 0.8)]
NSTEPS = [1, 2, 3, 5]


def gen_returns():
    import torch
    from rlpyt.algos.utils import (discount_return, generalized_advantage_estimation,
                                   discount_return_n_step, valid_from_done)
    out = {}
    for name, seed, T, B, p_done, sparse, pattern in RETURNS_CASES:
        if name == "kat":  # SURVEY.md 9.1 hand-checkable vector
            reward = np.array([[1, 0], [0, 2], [1, 1], [0.5, -1]], dtype=np.float32)
            value = np.array([[0.5, 0.1], [0.2, 0.3], [0.0, -0.2], [1.0, 0.4]], dtype=np.float32)
            done = np.array([[0, 0], [1, 0], [0, 0], [0, 1]], dtype=bool)
            bv = np.array([[2.0, 3.0]], dtype=np.float32)
        else:
            reward, value, done, bv = returns_inputs(seed, T, B, p_done, sparse, pattern)
        out[f"{name}/reward"], out[f"{name}/value"] = reward, value
        out[f"{name}/done"], out[f"{name}/bv"] = done, bv
        done_f = done.astype(np.float32)  # pg/base.py:51 casts done to reward dtype
        big = T * B > 8192  # keep the committed fixture small: fewer variants at full size
        for (g, lam) in (GAMMAS_LAMBDAS[:3] if big else GAMMAS_LAMBDAS):
            key = f"{name}/g{g}_l{lam}"
            # numpy path
            adv, ret = generalized_advantage_estimation(reward, value, done_f, bv, g, lam)
            # torch-CPU path (the one PPO really takes) must agree bit-for-bit
            adv_t, ret_t = generalized_advantage_estimation(
                torch.from_numpy(reward), torch.from_numpy(value), torch.from_numpy(done_f),
                torch.from_numpy(bv), g, lam)
            assert np.array_equal(adv, adv_t.numpy()) and np.array_equal(ret, ret_t.numpy())
            out[key + "/gae_adv"], out[key + "/gae_ret"] = adv, ret
            dr = discount_return(reward, done_f, bv, g)
            dr_t = discount_return(torch.from_numpy(reward), torch.from_numpy(done_f),
                                   torch.from_numpy(bv), g)
            assert np.array_equal(dr, dr_t.numpy())
            out[key + "/disc_ret"] = dr
        out[f"{name}/valid"] = valid_from_done(torch.from_numpy(done_f)).numpy()
        for n in ([3] if big else NSTEPS):
            for trunc in (False, True):
                if not trunc and T - (n - 1) < 1:
                    continue
                for g in ((0.99,) if big else (0.99, 0.5)):
                    r_, dn_ = discount_return_n_step(reward, done, n, g, do_truncated=trunc)
                    out[f"{name}/n{n}_t{int(trunc)}_g{g}/ret"] = np.asarray(r_, dtype=np.float32)
                    out[f"{name}/n{n}_t{int(trunc)}_g{g}/done_n"] = np.asarray(dn_)
    # process_returns through the reference PolicyGradientAlgo (normalisation, valid mask)
    from rlpyt.algos.pg.base import PolicyGradientAlgo
    from collections import namedtuple
    S = namedtuple("S", "env agent")
    E = namedtuple("E", "reward done")
    A = namedtuple("A", "agent_info bootstrap_value")
    I = namedtuple("I", "value")
    for name in ("cfg1", "edges", "ragged", "cfg2"):
        reward, value, done, bv = (out[f"{name}/{k}"] for k in ("reward", "value", "done", "bv"))
        samples = S(env=E(torch.from_numpy(reward), torch.from_numpy(done)),
                    agent=A(I(torch.from_numpy(value)), torch.from_numpy(bv)))
        for lam in ((0.98,) if name == "cfg2" else (1.0, 0.98)):
            for mid_batch_reset in (True, False):
                for norm in (False, True):
                    algo = PolicyGradientAlgo()
                    algo.discount, algo.gae_lambda = 0.99, lam
                    algo.normalize_advantage = norm
                    algo.mid_batch_reset = mid_batch_reset
                    algo.agent = types.SimpleNamespace(recurrent=False)
                    ret, adv, valid = algo.process_returns(samples)
                    key = f"{name}/pr_l{lam}_m{int(mid_batch_reset)}_n{int(norm)}"
                    out[key + "/ret"], out[key + "/adv"] = ret.numpy(), adv.numpy()
                    if valid is not None:
                        out[key + "/valid"] = valid.numpy()
    _save("returns", out)



# --------------------------------------------------------------------------- pg loss
def loss_inputs(seed, N, A, with_valid, zero_adv_frac=0.05):
    """Synthetic minibatch for the loss kernels (SURVEY.md 8(d) row 3: N=8192, A=6)."""
    rng = np.random.default_rng(seed)
    logits = rng.standard_normal((N, A)).astype(np.float32)
    e = np.exp(logits - logits.max(-1, keepdims=True))
    p_new = (e / e.sum(-1, keepdims=True)).astype(np.float32)
    logits_old = logits + 0.15 * rng.standard_normal((N, A)).astype(np.float32)
    e = np.exp(logits_old - logits_old.max(-1, keepdims=True))
    p_old = (e / e.sum(-1, keepdims=True)).astype(np.float32)
    same = rng.random(N) < 0.1          # ratio exactly 1 on some rows
    p_old[same] = p_new[same]
    value = rng.standard_normal(N).astype(np.float32)
    action = rng.integers(0, A, size=N).astype(np.int64)
    adv = rng.standard_normal(N).astype(np.float32)
    adv[rng.random(N) < zero_adv_frac] = 0.0
    ret = rng.standard_normal(N).astype(np.float32)
    valid = (rng.random(N) < 0.8).astype(np.float32) if with_valid else None
    return p_new, p_old, value, action, adv, ret, valid


LOSS_CASES = [
    # name, seed, N, A, with_valid, clip, c_v, c_ent
    ("kat", None, 4, 3, False, 0.1, 1.0, 0.01),
    ("kat_valid", None, 4, 3, True, 0.1, 1.0, 0.01),
    ("n37_a18", 21, 37, 18, False, 0.2, 0.5, 0.01),
    ("n37_a18_valid", 22, 37, 18, True, 0.2, 0.5, 0.01),
    ("a2c_cfg", 23, 1280, 6, False, 0.1, 0.5, 0.01),
    ("a2c_cfg_valid", 24, 1280, 6, True, 0.1, 0.5, 0.01),
    ("ppo_cfg", 25, 8192, 6, False, 0.1, 1.0, 0.01),
    ("ppo_cfg_valid", 26, 8192, 6, True, 0.1, 1.0, 0.01),
    ("n1", 27, 1, 4, False, 0.1, 1.0, 0.01),
]


def gen_loss():
    import torch
    from rlpyt.algos.pg.ppo import PPO
    from rlpyt.algos.pg.a2c import A2C
    from rlpyt.distributions.categorical import Categorical, DistInfo
    from rlpyt.agents.base import AgentInputs
    from collections import namedtuple

    class StubAgent:
        """Stands in for the network: returns fixed (prob, value) leaves so the reference's own
        PPO.loss / A2C.loss arithmetic and autograd run unmodified."""
        recurrent = False

        def __init__(self, p, v, A):
            self.p, self.v = p, v
            self.distribution = Categorical(dim=A)

        def __call__(self, observation, prev_action, prev_reward):
            return DistInfo(prob=self.p), self.v

    out = {}
    for name, seed, N, A, with_valid, clip, c_v, c_ent in LOSS_CASES:
        if name.startswith("kat"):  # SURVEY.md 9.2
            p_new = np.array([[.2, .5, .3], [.6, .3, .1], [.1, .1, .8], [.25, .25, .5]], np.float32)
            p_old = np.array([[.3, .4, .3], [.5, .4, .1], [.2, .2, .6], [.25, .25, .5]], np.float32)
            value = np.array([.5, -.2, 1, 0], np.float32)
            action = np.array([1, 0, 2, 1], np.int64)
            adv = np.array([1, -.5, 2, .3], np.float32)
            ret = np.array([1, 0, .5, -.4], np.float32)
            valid = np.array([1, 1, 0, 1], np.float32) if with_valid else None
        else:
            p_new, p_old, value, action, adv, ret, valid = loss_inputs(seed, N, A, with_valid)
        for k, x in dict(p_new=p_new, p_old=p_old, value=value, action=action, adv=adv, ret=ret).items():
            out[f"{name}/{k}"] = x
        if valid is not None:
            out[f"{name}/valid"] = valid
        out[f"{name}/hyper"] = np.array([clip, c_v, c_ent], np.float64)
        # ---- PPO.loss through the reference class
        p = torch.from_numpy(p_new).clone().requires_grad_(True)
        v = torch.from_numpy(value).clone().requires_grad_(True)
        algo = PPO(value_loss_coeff=c_v, entropy_loss_coeff=c_ent, ratio_clip=clip)
        algo.agent = StubAgent(p, v, A)
        dummy = AgentInputs(torch.zeros(N), torch.zeros(N), torch.zeros(N))
        loss, entropy, perplexity = algo.loss(
            dummy, torch.from_numpy(action), torch.from_numpy(ret), torch.from_numpy(adv),
            None if valid is None else torch.from_numpy(valid), DistInfo(prob=torch.from_numpy(p_old)))
        loss.backward()
        out[f"{name}/ppo/scalars"] = np.array([loss.item(), entropy.item(), perplexity.item()], np.float64)
        out[f"{name}/ppo/grad_prob"] = p.grad.numpy().copy()
        out[f"{name}/ppo/grad_value"] = v.grad.numpy().copy()
        # ---- A2C.loss: the reference method also calls process_returns(samples); feed it
        # pre-computed (return_, advantage, valid) by overriding that one method on the instance.
        p = torch.from_numpy(p_new).clone().requires_grad_(True)
        v = torch.from_numpy(value).clone().requires_grad_(True)
        a2c = A2C(value_loss_coeff=c_v, entropy_loss_coeff=c_ent)
        a2c.agent = StubAgent(p, v, A)
        a2c.process_returns = lambda samples: (torch.from_numpy(ret), torch.from_numpy(adv),
                                               None if valid is None else torch.from_numpy(valid))
        S = namedtuple("S", "env agent")
        E = namedtuple("E", "observation prev_reward")
        Ag = namedtuple("Ag", "prev_action action")
        samples = S(E(torch.zeros(N), torch.zeros(N)), Ag(torch.zeros(N), torch.from_numpy(action)))
        loss, entropy, perplexity = a2c.loss(samples)
        loss.backward()
        out[f"{name}/a2c/scalars"] = np.array([loss.item(), entropy.item(), perplexity.item()], np.float64)
        out[f"{name}/a2c/grad_prob"] = p.grad.numpy().copy()
        out[f"{name}/a2c/grad_value"] = v.grad.numpy().copy()
    _save("loss", out)


# --------------------------------------------------------------------------- PPO / A2C iteration
def rollout_inputs(seed, T, B, image_shape, A):
    """A synthetic [T,B] batch as the sampler would hand it to the algorithm."""
    rng = np.random.default_rng(seed)
    obs = rng.integers(0, 256, size=(T, B) + tuple(image_shape), dtype=np.uint8)
    action = rng.integers(0, A, size=(T, B)).astype(np.int64)
    reward = rng.choice(np.array([-1, 0, 1], np.float32), size=(T, B), p=[0.1, 0.8, 0.1]).astype(np.float32)
    done = rng.random((T, B)) < 0.05
    value = rng.standard_normal((T, B)).astype(np.float32) * 0.1
    logits = rng.standard_normal((T, B, A)).astype(np.float32) * 0.3
    e = np.exp(logits - logits.max(-1, keepdims=True))
    old_prob = (e / e.sum(-1, keepdims=True)).astype(np.float32)
    bv = rng.standard_normal((1, B)).astype(np.float32) * 0.1
    return obs, action, reward, done, value, old_prob, bv


def gen_ppo():
    """Two iterations of the reference PPO / one of A2C on a tiny AtariFf problem, CPU."""
    import torch
    from collections import namedtuple
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import atari_ff
    from rlpyt.algos.pg.ppo import PPO
    from rlpyt.algos.pg.a2c import A2C
    from rlpyt.agents.pg.atari import AtariFfAgent
    from rlpyt.samplers.collections import Samples, AgentSamplesBsv, EnvSamples, BatchSpec
    from rlpyt.agents.pg.base import AgentInfo
    from rlpyt.distributions.categorical import DistInfo
    Spaces = namedtuple("Spaces", "observation action")
    Obs = namedtuple("Obs", "shape")
    Act = namedtuple("Act", "n")
    out = {}
    T, B, image_shape, A = 8, 6, (4, 36, 36), 5
    torch.set_num_threads(1)
    for algo_name in ("ppo", "ppo_valid_norm", "a2c"):
        sd0 = atari_ff.init_state_dict(image_shape, A, seed=3)
        agent = AtariFfAgent(initial_model_state_dict={k: v.clone() for k, v in sd0.items()})
        agent.initialize(Spaces(Obs(image_shape), Act(A)))
        n_itr = 4
        if algo_name == "a2c":
            algo = A2C(gae_lambda=0.95, normalize_advantage=False)
        elif algo_name == "ppo":
            algo = PPO(gae_lambda=0.98, minibatches=2, epochs=2)
        else:
            algo = PPO(gae_lambda=1, minibatches=3, epochs=2, normalize_advantage=True, ratio_clip=0.2)
        mbr = algo_name != "ppo_valid_norm"
        algo.initialize(agent, n_itr, BatchSpec(T, B), mid_batch_reset=mbr)
        np.random.seed(77)
        out[f"{algo_name}/sd0_seed"] = np.array([3])  # atari_ff.init_state_dict(image_shape, A, seed=3)
        out[f"{algo_name}/sd0_check"] = np.array([float(sum(v.double().sum() for v in sd0.values()))])
        for itr in range(2):
            obs, action, reward, done, value, old_prob, bv = rollout_inputs(100 + itr, T, B, image_shape, A)
            for k, x in dict(obs=obs, action=action, reward=reward, done=done, value=value,
                             old_prob=old_prob, bv=bv).items():
                out[f"{algo_name}/itr{itr}/{k}"] = x
            t = torch.from_numpy
            all_action = torch.cat([torch.zeros(1, B, dtype=torch.int64), t(action)])
            all_reward = torch.cat([torch.zeros(1, B), t(reward)])
            samples = Samples(
                agent=AgentSamplesBsv(action=all_action[1:], prev_action=all_action[:-1],
                                      agent_info=AgentInfo(dist_info=DistInfo(prob=t(old_prob)), value=t(value)),
                                      bootstrap_value=t(bv)),
                env=EnvSamples(observation=t(obs), reward=all_reward[1:], prev_reward=all_reward[:-1],
                               done=t(done), env_info=None))
            agent.train_mode(itr)
            info = algo.optimize_agent(itr, samples)
            for f in ("loss", "gradNorm", "entropy", "perplexity"):
                out[f"{algo_name}/itr{itr}/opt_{f}"] = np.atleast_1d(np.asarray(getattr(info, f), np.float64))
            for k, v in agent.state_dict().items():  # fc weight: first 8 rows only (fixture size)
                a = v.detach().numpy().copy()
                out[f"{algo_name}/itr{itr}/sd/{k}"] = a[:8] if k == "conv.head.model.0.weight" else a
    _save("ppo", out)


def gen_ppo_lstm():
    """Two iterations of the reference's RECURRENT PPO (AtariLstmAgent, whole trajectories, minibatches over B, valid
    mask) and one of recurrent A2C on a tiny problem, CPU.  The initial weights are stored (LSTM included)."""
    import torch
    from collections import namedtuple
    from rlpyt.algos.pg.ppo import PPO
    from rlpyt.algos.pg.a2c import A2C
    from rlpyt.agents.pg.atari import AtariLstmAgent
    from rlpyt.agents.pg.base import AgentInfoRnn
    from rlpyt.distributions.categorical import DistInfo
    from rlpyt.models.pg.atari_lstm_model import RnnState
    from rlpyt.samplers.collections import Samples, AgentSamplesBsv, EnvSamples, BatchSpec
    Spaces = namedtuple("Spaces", "observation action")
    Obs = namedtuple("Obs", "shape")
    Act = namedtuple("Act", "n")
    out = {}
    T, B, image_shape, A, H = 8, 6, (4, 36, 36), 5, 64
    torch.set_num_threads(1)
    for algo_name in ("ppo", "a2c"):
        torch.manual_seed(5)
        agent = AtariLstmAgent(model_kwargs=dict(fc_sizes=128, lstm_size=H))
        agent.initialize(Spaces(Obs(image_shape), Act(A)))
        for k, v in agent.state_dict().items():
            out[f"{algo_name}/sd0/{k}"] = v.detach().numpy().copy()
        algo = PPO(gae_lambda=0.95, minibatches=2, epochs=2) if algo_name == "ppo" else A2C(gae_lambda=0.95)
        algo.initialize(agent, 4, BatchSpec(T, B), mid_batch_reset=True)
        np.random.seed(78)
        for itr in range(2):
            obs, action, reward, done, value, old_prob, bv = rollout_inputs(200 + itr, T, B, image_shape, A)
            rng = np.random.default_rng(300 + itr)
            h0 = (rng.standard_normal((T, B, 1, H)) * 0.1).astype(np.float32)      # recorded [T,B,N,H]; only [0] is used
            c0 = (rng.standard_normal((T, B, 1, H)) * 0.1).astype(np.float32)
            for k, x in dict(obs=obs, action=action, reward=reward, done=done, value=value, old_prob=old_prob, bv=bv,
                             h0=h0, c0=c0).items():
                out[f"{algo_name}/itr{itr}/{k}"] = x
            t = torch.from_numpy
            all_action = torch.cat([torch.zeros(1, B, dtype=torch.int64), t(action)])
            all_reward = torch.cat([torch.zeros(1, B), t(reward)])
            samples = Samples(
                agent=AgentSamplesBsv(action=all_action[1:], prev_action=all_action[:-1],
                                      agent_info=AgentInfoRnn(dist_info=DistInfo(prob=t(old_prob)), value=t(value),
                                                              prev_rnn_state=RnnState(h=t(h0), c=t(c0))),
                                      bootstrap_value=t(bv)),
                env=EnvSamples(observation=t(obs), reward=all_reward[1:], prev_reward=all_reward[:-1],
                               done=t(done), env_info=None))
            agent.train_mode(itr)
            info = algo.optimize_agent(itr, samples)
            for f in ("loss", "gradNorm", "entropy", "perplexity"):
                out[f"{algo_name}/itr{itr}/opt_{f}"] = np.atleast_1d(np.asarray(getattr(info, f), np.float64))
            if algo_name == "a2c":
                break
    _save("ppo_lstm", out)


# --------------------------------------------------------------------------- replay
def replay_stream(seed, n_batches, T, B, obs_shape, A, p_done):
    """Consecutive sampler batches with proper frame history (frame c of step t = frame c+1 of t-1)."""
    rng = np.random.default_rng(seed)
    nf = obs_shape[0]
    hist = rng.integers(0, 256, size=(nf - 1, B) + tuple(obs_shape[1:]), dtype=np.uint8)
    for _ in range(n_batches):
        new = rng.integers(0, 256, size=(T, B) + tuple(obs_shape[1:]), dtype=np.uint8)
        full = np.concatenate([hist, new], 0)                       # [T+nf-1,B,H,W]
        obs = np.stack([full[c:c + T] for c in range(nf)], axis=2)   # [T,B,nf,H,W]
        hist = full[-(nf - 1):] if nf > 1 else hist
        yield dict(observation=obs, action=rng.integers(0, A, size=(T, B)).astype(np.int64),
                   reward=rng.standard_normal((T, B)).astype(np.float32), done=rng.random((T, B)) < p_done)


REPLAY_CASES = [
    # name, seed, size, B, obs_shape, n_step, discount, batch_T, n_batches, batch_B, prioritized, unique
    ("kat", 31, 16, 2, (3, 1, 1), 2, 0.5, 4, 6, 5, True, False),
    ("small_pri", 32, 96, 4, (4, 6, 5), 3, 0.99, 5, 9, 16, True, False),
    ("small_pri_unique", 33, 96, 4, (4, 6, 5), 3, 0.99, 5, 9, 12, True, True),
    ("small_uni", 34, 96, 4, (4, 6, 5), 3, 0.99, 5, 9, 16, False, False),
    ("n1_f1", 35, 60, 3, (1, 4, 4), 1, 0.9, 7, 6, 10, True, False),
    ("mid_pri", 36, 2048, 8, (4, 12, 12), 3, 0.99, 16, 24, 64, True, False),
    ("bigT_append", 37, 64, 4, (2, 3, 3), 5, 0.95, 13, 5, 8, True, False),
]


def gen_replay():
    import torch
    from rlpyt.replays.non_sequence.frame import PrioritizedReplayFrameBuffer, UniformReplayFrameBuffer
    from rlpyt.replays.sum_tree import SumTree
    from rlpyt.algos.dqn.dqn import SamplesToBuffer
    from rlpyt.utils.logging import logger
    logger.log = lambda *a, **k: None
    out = {}
    for (name, seed, size, B, obs_shape, n_step, discount, batch_T, n_batches, batch_B, prioritized,
         unique) in REPLAY_CASES:
        example = SamplesToBuffer(observation=np.zeros(obs_shape, np.uint8), action=np.int64(0),
                                  reward=np.float32(0), done=np.bool_(False))
        kw = dict(example=example, size=size, B=B, discount=discount, n_step_return=n_step)
        buf = (PrioritizedReplayFrameBuffer(alpha=0.6, beta=0.4, default_priority=1, unique=unique, **kw)
               if prioritized else UniformReplayFrameBuffer(**kw))
        out[f"{name}/cfg"] = np.array([seed, size, B, n_step, batch_T, n_batches, batch_B, int(prioritized), int(unique)])
        out[f"{name}/obs_shape"] = np.array(obs_shape)
        out[f"{name}/discount"] = np.array([discount])
        np.random.seed(seed)
        rng = np.random.default_rng(seed + 1000)
        for i, s in enumerate(replay_stream(seed, n_batches, batch_T, B, obs_shape, 4, 0.1)):
            buf.append_samples(SamplesToBuffer(**s))
            out[f"{name}/b{i}/t"] = np.array([buf.t])
            if prioritized:
                out[f"{name}/b{i}/root"] = np.array([buf.priority_tree.tree[0]])
            if i < 2:  # too early to sample (nothing valid yet in tiny buffers)
                continue
            if prioritized and buf.priority_tree.tree[0] <= 0:
                continue
            u = rng.random(batch_B)
            if prioritized:
                if unique:
                    batch = buf.sample_batch(batch_B)      # draws from np.random internally
                else:
                    state = np.random.get_state()
                    np.random.rand(batch_B)                 # keep the stream position of sample()
                    np.random.set_state(state)
                    import rlpyt.replays.sum_tree as st
                    orig = np.random.rand
                    st.np.random.rand = lambda n, _u=u: _u.copy()   # inject known uniforms
                    try:
                        batch = buf.sample_batch(batch_B)
                    finally:
                        st.np.random.rand = orig
                    out[f"{name}/b{i}/uniforms"] = u
                tidx = buf.priority_tree.prev_tree_idxs
                out[f"{name}/b{i}/tree_idxs"] = np.asarray(tidx).copy()
                out[f"{name}/b{i}/is_weights"] = batch.is_weights.numpy().copy()
            else:
                st0 = np.random.get_state()
                batch = buf.sample_batch(batch_B)
                np.random.set_state(st0)
                T_idxs, B_idxs = buf.sample_idxs(batch_B)
                out[f"{name}/b{i}/T_idxs"], out[f"{name}/b{i}/B_idxs"] = T_idxs, B_idxs
            flat = dict(observation=batch.agent_inputs.observation, prev_action=batch.agent_inputs.prev_action,
                        prev_reward=batch.agent_inputs.prev_reward, action=batch.action, return_=batch.return_,
                        done=batch.done, done_n=batch.done_n, target_observation=batch.target_inputs.observation,
                        target_prev_action=batch.target_inputs.prev_action,
                        target_prev_reward=batch.target_inputs.prev_reward)
            for k, v in flat.items():
                out[f"{name}/b{i}/{k}"] = v.numpy().copy()
            if prioritized:
                new_pri = np.abs(rng.standard_normal(batch_B)).astype(np.float32) + 0.01
                out[f"{name}/b{i}/new_pri"] = new_pri
                buf.update_batch_priorities(torch.from_numpy(new_pri))
                out[f"{name}/b{i}/root_after"] = np.array([buf.priority_tree.tree[0]])
        if prioritized:
            out[f"{name}/final_tree"] = buf.priority_tree.tree.copy()
        out[f"{name}/final_frames"] = buf.samples_frames.copy() if buf.samples_frames.size < 200000 else buf.samples_frames[:8].copy()
        out[f"{name}/final_return"] = buf.samples_return_.copy()
        out[f"{name}/final_done_n"] = buf.samples_done_n.copy()
    # raw SumTree known answers of SURVEY.md 9.3
    tree = SumTree(T=6, B=2, off_backward=2, off_forward=1, default_value=1.0)
    for k in range(5):
        tree.advance(2)
        out[f"tree_kat/adv{k}"] = tree.tree.copy()
    np.random.seed(3)
    (T_idxs, B_idxs), pri = tree.sample(5)
    out["tree_kat/T_idxs"], out["tree_kat/B_idxs"], out["tree_kat/pri"] = T_idxs, B_idxs, pri
    tree.update_batch_priorities(np.array([0.5, 2.0, 3.0, 0.25, 4.0]))
    out["tree_kat/after_update"] = tree.tree.copy()
    idx, _ = tree.find(np.array([0, 0.1, 0.5, 0.999999, 1.0]))
    out["tree_kat/find"] = idx
    _save("replay", out)


# --------------------------------------------------------------------------- sequence replay (R2D1)
SEQ_REPLAY_CASES = [
    # name, seed, size, B, obs_shape, n_step, discount, sampler_T, n_batches, batch_B, batch_T, rsi, prioritized,
    # input_priorities, input_priority_shift
    ("seq_uni_norn", 51, 96, 4, (4, 5, 4), 3, 0.99, 6, 9, 12, 5, 0, False, False, 0),
    ("seq_uni_rsi1", 52, 96, 4, (4, 5, 4), 2, 0.9, 6, 9, 12, 4, 1, False, False, 0),
    ("seq_uni_rsi4", 53, 128, 4, (3, 4, 4), 3, 0.99, 8, 9, 10, 8, 4, False, False, 0),
    ("seq_pri_rsi1", 54, 96, 4, (4, 5, 4), 3, 0.99, 6, 9, 12, 5, 1, True, False, 0),
    ("seq_pri_rsi4_input", 55, 128, 4, (4, 4, 4), 3, 0.997, 4, 16, 8, 8, 4, True, True, 1),
    ("seq_pri_norn", 56, 60, 3, (2, 3, 3), 1, 0.95, 5, 8, 7, 3, 0, True, False, 0),
    ("seq_mid", 57, 2048, 8, (4, 6, 6), 5, 0.997, 16, 20, 8, 24, 8, True, True, 1),
]


def gen_seq_replay():
    import torch
    from rlpyt.replays.sequence.frame import (PrioritizedSequenceReplayFrameBuffer,
                                              UniformSequenceReplayFrameBuffer)
    from rlpyt.algos.dqn.dqn import SamplesToBuffer
    from rlpyt.algos.dqn.r2d1 import SamplesToBufferRnn, PrioritiesSamplesToBuffer
    from rlpyt.utils.collections import namedarraytuple
    RnnState = namedarraytuple("RnnState", ["h", "c"])
    out = {}
    for (name, seed, size, B, obs_shape, n_step, discount, sampler_T, n_batches, batch_B, batch_T, rsi, prioritized,
         input_pri, pri_shift) in SEQ_REPLAY_CASES:
        example = SamplesToBuffer(observation=np.zeros(obs_shape, np.uint8), action=np.int64(0),
                                  reward=np.float32(0), done=np.bool_(False))
        if rsi > 0:
            example = SamplesToBufferRnn(*example, prev_rnn_state=RnnState(h=np.zeros((1, 3), np.float32),
                                                                           c=np.zeros((1, 3), np.float32)))
        kw = dict(example=example, size=size, B=B, discount=discount, n_step_return=n_step, rnn_state_interval=rsi,
                  batch_T=batch_T)
        if prioritized:
            buf = PrioritizedSequenceReplayFrameBuffer(alpha=0.6, beta=0.9, default_priority=1, unique=False,
                                                       input_priorities=input_pri, input_priority_shift=pri_shift, **kw)
        else:
            buf = UniformSequenceReplayFrameBuffer(**kw)
        out[f"{name}/cfg"] = np.array([seed, size, B, n_step, sampler_T, n_batches, batch_B, batch_T, rsi, int(prioritized),
                                       int(input_pri), pri_shift])
        out[f"{name}/obs_shape"] = np.array(obs_shape)
        out[f"{name}/discount"] = np.array([discount])
        out[f"{name}/T"] = np.array([buf.T])
        np.random.seed(seed)
        rng = np.random.default_rng(seed + 1000)
        for i, s in enumerate(replay_stream(seed, n_batches, sampler_T, B, obs_shape, 4, 0.08)):
            stb = SamplesToBuffer(**s)
            if rsi > 0:
                rnn = RnnState(h=rng.standard_normal((sampler_T, B, 1, 3)).astype(np.float32),
                               c=rng.standard_normal((sampler_T, B, 1, 3)).astype(np.float32))
                out[f"{name}/b{i}/rnn_h"], out[f"{name}/b{i}/rnn_c"] = rnn.h, rnn.c
                stb = SamplesToBufferRnn(*stb, prev_rnn_state=rnn)
            if input_pri:
                pri = (np.abs(rng.standard_normal(B)) + 0.05).astype(np.float32)      # [B], as R2D1.compute_input_priorities
                out[f"{name}/b{i}/input_pri"] = pri
                stb = PrioritiesSamplesToBuffer(priorities=pri, samples=stb)
            buf.append_samples(stb)
            out[f"{name}/b{i}/t"] = np.array([buf.t])
            if prioritized:
                out[f"{name}/b{i}/root"] = np.array([buf.priority_tree.tree[0]])
            enough = buf._buffer_full or buf.t > batch_T + n_step + max(1, obs_shape[0] - 1) + max(1, rsi)
            if not enough or (prioritized and buf.priority_tree.tree[0] <= 0):
                continue
            if prioritized:
                u = rng.random(batch_B)
                import rlpyt.replays.sum_tree as st
                orig = np.random.rand
                st.np.random.rand = lambda n, _u=u: _u.copy()
                try:
                    batch = buf.sample_batch(batch_B)
                finally:
                    st.np.random.rand = orig
                out[f"{name}/b{i}/uniforms"] = u
                out[f"{name}/b{i}/tree_idxs"] = np.asarray(buf.priority_tree.prev_tree_idxs).copy()
                out[f"{name}/b{i}/is_weights"] = batch.is_weights.numpy().copy()
            else:
                st0 = np.random.get_state()
                batch = buf.sample_batch(batch_B)
                np.random.set_state(st0)
                T_idxs, B_idxs = buf.sample_idxs(batch_B, batch_T)
                out[f"{name}/b{i}/T_idxs"], out[f"{name}/b{i}/B_idxs"] = T_idxs, B_idxs
            for k in ("all_observation", "all_action", "all_reward", "return_", "done", "done_n"):
                out[f"{name}/b{i}/{k}"] = getattr(batch, k).numpy().copy()
            if rsi > 0:
                out[f"{name}/b{i}/init_h"] = batch.init_rnn_state.h.numpy().copy()
                out[f"{name}/b{i}/init_c"] = batch.init_rnn_state.c.numpy().copy()
            if prioritized:
                new_pri = np.abs(rng.standard_normal(batch_B)).astype(np.float32) + 0.01
                out[f"{name}/b{i}/new_pri"] = new_pri
                buf.update_batch_priorities(torch.from_numpy(new_pri))
                out[f"{name}/b{i}/root_after"] = np.array([buf.priority_tree.tree[0]])
        if prioritized:
            out[f"{name}/final_tree"] = buf.priority_tree.tree.copy()
        out[f"{name}/final_return"] = buf.samples_return_.copy()
        out[f"{name}/final_done_n"] = buf.samples_done_n.copy()
        if rsi > 1:
            out[f"{name}/final_rnn_h"] = buf.samples_prev_rnn_state.h.copy()
    # extract_sequences known answers, including the wrap-at-the-beginning placement (misc.py:49-51)
    from rlpyt.utils.misc import extract_sequences
    arr = np.arange(10 * 3).reshape(10, 3)
    out["extract_kat/arr"] = arr
    out["extract_kat/T_idxs"] = np.array([-1, 0, 7, 8, 9, -2, 3])
    out["extract_kat/B_idxs"] = np.array([0, 1, 2, 0, 1, 2, 0])
    out["extract_kat/out"] = extract_sequences(arr, out["extract_kat/T_idxs"], out["extract_kat/B_idxs"], 4)
    _save("seq_replay", out)


# --------------------------------------------------------------------------- R2D1
R2D1_CASES = [
    # name, seed, wT, bT, n_step, B, double, prioritized, delta_clip, rsi, dueling
    ("r2d1_double_pri", 61, 4, 6, 3, 5, True, True, None, 2, False),
    ("r2d1_plain_uniform_huber", 62, 0, 7, 1, 4, False, False, 1.0, 0, False),
    ("r2d1_dueling", 63, 3, 5, 2, 6, True, True, None, 1, True),
]


def gen_r2d1():
    """R2D1.loss (warm-up, double-Q, value rescaling, valid masks, sequence priorities) and compute_input_priorities of the
    reference on a tiny AtariR2d1Model, CPU: the initial weights of both networks, the sampled batch, the loss, the TD
    errors, the priorities and the gradient of every parameter."""
    import torch
    from collections import namedtuple
    from rlpyt.algos.dqn.r2d1 import R2D1
    from rlpyt.agents.dqn.atari.atari_r2d1_agent import AtariR2d1Agent
    from rlpyt.models.dqn.atari_r2d1_model import RnnState
    from rlpyt.replays.sequence.prioritized import SamplesFromReplayPri
    from rlpyt.replays.sequence.n_step import SamplesFromReplay
    from rlpyt.samplers.collections import Samples, AgentSamples, EnvSamples
    from rlpyt.agents.dqn.r2d1_agent import AgentInfo
    Spaces = namedtuple("Spaces", "observation action")
    Obs = namedtuple("Obs", "shape")
    Act = namedtuple("Act", "n")
    out = {}
    image_shape, A, H = (4, 36, 36), 5, 16
    torch.set_num_threads(1)
    for (name, seed, wT, bT, n, B, double, prioritized, delta_clip, rsi, dueling) in R2D1_CASES:
        torch.manual_seed(seed)
        agent = AtariR2d1Agent(model_kwargs=dict(channels=[4, 8, 8], fc_size=32, lstm_size=H, head_size=16, dueling=dueling))
        agent.initialize(Spaces(Obs(image_shape), Act(A)))
        with torch.no_grad():                                     # make the target network differ from the online one
            for p_ in agent.target_model.parameters():
                p_.add_(0.05 * torch.randn_like(p_))
        for k, v in agent.model.state_dict().items():
            out[f"{name}/model/{k}"] = v.detach().numpy().copy()
        for k, v in agent.target_model.state_dict().items():
            out[f"{name}/target/{k}"] = v.detach().numpy().copy()
        algo = R2D1(discount=0.99, batch_T=bT, batch_B=B, warmup_T=wT, store_rnn_state_interval=rsi, n_step_return=n,
                    double_dqn=double, prioritized_replay=prioritized, delta_clip=delta_clip, pri_eta=0.9,
                    input_priority_shift=0 if rsi == 0 else None)
        algo.agent = agent
        rng = np.random.default_rng(seed)
        L = wT + bT + n
        batch = dict(
            all_observation=rng.integers(0, 256, size=(L, B) + image_shape, dtype=np.uint8),
            all_action=rng.integers(0, A, size=(L, B)).astype(np.int64),
            all_reward=(rng.standard_normal((L, B)) * 3).astype(np.float32),        # beyond +-1: the value rescaling matters
            return_=(rng.standard_normal((wT + bT, B)) * 4).astype(np.float32),
            done=rng.random((wT + bT, B)) < 0.08,
            done_n=rng.random((wT + bT, B)) < 0.15,
            init_h=(rng.standard_normal((B, 1, H)) * 0.3).astype(np.float32),
            init_c=(rng.standard_normal((B, 1, H)) * 0.3).astype(np.float32),
            is_weights=(rng.random(B) * 0.8 + 0.2).astype(np.float32),
        )
        if wT > 0:
            batch["done"][wT - 1, 1] = True                        # a trajectory that ends inside the warm-up (state reset)
        batch["done"][wT + 2, 0] = True                            # and one inside the training segment (valid mask)
        cfg = np.array([seed, wT, bT, n, B, int(double), int(prioritized), -1.0 if delta_clip is None else delta_clip, rsi,
                        int(dueling), A, H])
        out[f"{name}/cfg"] = cfg
        for k, v in batch.items():
            if k != "all_observation":      # the first draw of default_rng(seed): the test regenerates it (fixture size)
                out[f"{name}/batch/{k}"] = v
        out[f"{name}/batch/all_observation_sum"] = np.array([batch["all_observation"].astype(np.int64).sum()])
        t = torch.from_numpy
        init = None if rsi == 0 else RnnState(h=t(batch["init_h"]), c=t(batch["init_c"]))
        base = SamplesFromReplay(all_observation=t(batch["all_observation"]), all_action=t(batch["all_action"]),
                                 all_reward=t(batch["all_reward"]), return_=t(batch["return_"]), done=t(batch["done"]),
                                 done_n=t(batch["done_n"]), init_rnn_state=init)
        samples = SamplesFromReplayPri(*base, is_weights=t(batch["is_weights"])) if prioritized else base
        agent.train_mode(0)
        loss, td, pri = algo.loss(samples)
        loss.backward()
        out[f"{name}/loss"] = np.array([loss.item()], np.float64)
        out[f"{name}/td_abs_errors"] = td.numpy().copy()
        out[f"{name}/priorities"] = pri.detach().numpy().copy()
        for k, p_ in agent.model.named_parameters():
            out[f"{name}/grad/{k}"] = (p_.grad if p_.grad is not None else torch.zeros_like(p_)).numpy().copy()
        # input priorities of a fresh sampler batch
        Ts = 9
        q = (rng.standard_normal((Ts, B, A)) * 2).astype(np.float32)
        act = rng.integers(0, A, size=(Ts, B)).astype(np.int64)
        rew = (rng.standard_normal((Ts, B)) * 2).astype(np.float32)
        dn = rng.random((Ts, B)) < 0.1
        smp = Samples(agent=AgentSamples(action=t(act), prev_action=t(act), agent_info=AgentInfo(q=t(q), prev_rnn_state=None)),
                      env=EnvSamples(observation=None, reward=t(rew), prev_reward=t(rew), done=t(dn), env_info=None))
        out[f"{name}/input/q"], out[f"{name}/input/action"] = q, act
        out[f"{name}/input/reward"], out[f"{name}/input/done"] = rew, dn
        if n > 1:      # (with n_step_return == 1 the reference's shapes do not line up, r2d1.py:216-219)
            out[f"{name}/input/priorities"] = np.asarray(algo.compute_input_priorities(smp)).copy()
    x = torch.tensor([-300., -7.5, -1., -1e-3, 0., 1e-3, 0.5, 1., 12., 4000.])
    algo = R2D1()
    out["value_scale/x"] = x.numpy()
    out["value_scale/h"] = algo.value_scale(x).numpy()
    out["value_scale/h_inv"] = algo.inv_value_scale(x).numpy()
    _save("r2d1", out)


# --------------------------------------------------------------------------- DQN loss
DQN_CASES = [
    # name, seed, N, A, double_dqn, prioritized, delta_clip, n_step, discount
    ("dqn_small", 40, 7, 4, False, False, 1.0, 1, 0.99),
    ("dqn_double_pri", 41, 512, 6, True, True, 1.0, 3, 0.99),
    ("dqn_pri", 42, 512, 6, False, True, 1.0, 3, 0.99),
    ("dqn_mse", 43, 33, 18, True, False, None, 1, 0.997),
    ("dqn_clip_frac", 44, 257, 9, True, True, 0.1, 5, 0.95),
    ("dqn_n1", 45, 1, 2, False, True, 1.0, 1, 0.99),
]


def dqn_inputs(seed, N, A):
    """Q-values with ties (argmax/first-index semantics), |delta| on both sides of the clip and exactly on it."""
    rng = np.random.default_rng(seed)
    qs = (rng.standard_normal((N, A)) * 1.5).astype(np.float32)
    target_qs = (rng.standard_normal((N, A)) * 1.5).astype(np.float32)
    next_qs = (rng.standard_normal((N, A)) * 1.5).astype(np.float32)
    if N > 4:
        next_qs[1, :] = next_qs[1, 0]                    # all equal: argmax -> 0
        next_qs[2, -1] = next_qs[2].max()                # duplicate maximum at the end
        target_qs[3, :] = target_qs[3, 0]
    action = rng.integers(0, A, size=N).astype(np.int64)
    return_ = rng.standard_normal(N).astype(np.float32)
    done_n = rng.random(N) < 0.1
    is_weights = rng.random(N).astype(np.float32) * 0.9 + 0.1
    if N > 6:                                            # |delta| == delta_clip exactly and delta == 0
        done_n[5], done_n[6] = True, True
        return_[5] = qs[5, action[5]] + np.float32(1.0)
        return_[6] = qs[6, action[6]]
    return qs, target_qs, next_qs, action, return_, done_n, is_weights


def gen_dqn():
    import torch
    from rlpyt.algos.dqn.dqn import DQN
    from rlpyt.agents.base import AgentInputs
    from collections import namedtuple

    class StubAgent:
        """Fixed network outputs: the reference's DQN.loss arithmetic and autograd run unmodified.
        The online net is called first on agent_inputs (tag 0), then on target_inputs (tag 1)."""

        def __init__(self, qs, next_qs, target_qs):
            self.qs, self.next_qs, self.target_qs = qs, next_qs, target_qs

        def __call__(self, observation, prev_action, prev_reward):
            return self.qs if int(observation[0]) == 0 else self.next_qs

        def target(self, observation, prev_action, prev_reward):
            return self.target_qs

    Samples = namedtuple("Samples", "agent_inputs action return_ done done_n target_inputs is_weights")
    out = {}
    for name, seed, N, A, double, pri, clip, n_step, discount in DQN_CASES:
        qs, target_qs, next_qs, action, return_, done_n, is_weights = dqn_inputs(seed, N, A)
        for k, x in dict(qs=qs, target_qs=target_qs, next_qs=next_qs, action=action, return_=return_,
                         done_n=done_n, is_weights=is_weights).items():
            out[f"{name}/{k}"] = x
        out[f"{name}/hyper"] = np.array([float(double), float(pri), -1.0 if clip is None else clip, n_step, discount],
                                        np.float64)
        q = torch.from_numpy(qs).clone().requires_grad_(True)
        algo = DQN(discount=discount, delta_clip=clip, n_step_return=n_step, double_dqn=double,
                   prioritized_replay=pri)
        algo.mid_batch_reset = True
        algo.agent = StubAgent(q, torch.from_numpy(next_qs), torch.from_numpy(target_qs))
        tag0 = AgentInputs(torch.zeros(N), torch.zeros(N), torch.zeros(N))
        tag1 = AgentInputs(torch.ones(N), torch.zeros(N), torch.zeros(N))
        samples = Samples(tag0, torch.from_numpy(action), torch.from_numpy(return_), torch.from_numpy(done_n),
                          torch.from_numpy(done_n), tag1, torch.from_numpy(is_weights))
        loss, td_abs = algo.loss(samples)
        loss.backward()
        out[f"{name}/loss"] = np.array([loss.item()], np.float64)
        out[f"{name}/td_abs_errors"] = td_abs.numpy().copy()
        out[f"{name}/grad_qs"] = q.grad.numpy().copy()
    _save("dqn", out)


def gen_collector():
    """The reference's own samplers (GpuSampler with cuda_idx=None, SerialSampler with the CPU collector) stepping
    the synthetic Atari-shaped env under the deterministic policy of tests/deterministic_agent.py: every field of
    the [T,B] batch for three consecutive iterations.  Pins oracle/collector.py and is what the GPU samplers are
    compared with (tests/test_gpu_sampler.py)."""
    import torch
    sys.path.insert(0, os.path.dirname(HERE))                     # tests/
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))    # repo root (baseline.reference_arm: the env)
    from deterministic_agent import make_agent_class
    from baseline.reference_arm import make_env_cls
    from rlpyt.agents.base import AgentStep
    from rlpyt.agents.pg.base import AgentInfo
    from rlpyt.distributions.categorical import DistInfo
    from rlpyt.samplers.parallel.gpu.sampler import GpuSampler
    from rlpyt.samplers.serial.sampler import SerialSampler
    from rlpyt.samplers.parallel.cpu.collectors import CpuResetCollector
    from rlpyt.samplers.parallel.gpu.collectors import GpuWaitResetCollector
    Agent = make_agent_class(AgentStep, AgentInfo, DistInfo)
    Env = make_env_cls()
    T, B, A, image = 6, 8, 5, (4, 36, 36)
    env_kwargs = dict(image_shape=image, n_actions=A, p_done=0.15, p_reward=0.4)
    out = {"T": np.array([T]), "B": np.array([B]), "A": np.array([A]), "image": np.array(image), "seed": np.array([11]),
           "p_done": np.array([0.15]), "p_reward": np.array([0.4])}
    cases = {
        "gpu": (GpuSampler, dict()),
        "gpu_wait_reset": (GpuSampler, dict(CollectorCls=GpuWaitResetCollector)),
        "serial": (SerialSampler, dict(CollectorCls=CpuResetCollector)),
    }
    for name, (Cls, extra) in cases.items():
        sampler = Cls(EnvCls=Env, env_kwargs=env_kwargs, batch_T=T, batch_B=B, max_decorrelation_steps=0, **extra)
        agent = Agent()
        affinity = dict(cuda_idx=None, workers_cpus=[0, 1], set_affinity=False)
        sampler.initialize(agent=agent, affinity=affinity, seed=11, bootstrap_value=True, traj_info_kwargs=dict(discount=0.99))
        for itr in range(3):
            agent.sample_mode(itr)
            samples, traj_infos = sampler.obtain_samples(itr)
            pre = f"{name}/itr{itr}/"
            out[pre + "observation"] = samples.env.observation.numpy().copy()
            out[pre + "reward"] = samples.env.reward.numpy().copy()
            out[pre + "prev_reward"] = samples.env.prev_reward.numpy().copy()
            out[pre + "done"] = samples.env.done.numpy().copy()
            out[pre + "traj_done"] = samples.env.env_info.traj_done.numpy().copy()
            out[pre + "game_score"] = samples.env.env_info.game_score.numpy().copy()
            out[pre + "action"] = samples.agent.action.numpy().copy()
            out[pre + "prev_action"] = samples.agent.prev_action.numpy().copy()
            out[pre + "prob"] = samples.agent.agent_info.dist_info.prob.numpy().copy()
            out[pre + "value"] = samples.agent.agent_info.value.numpy().copy()
            out[pre + "bootstrap_value"] = samples.agent.bootstrap_value.numpy().copy()
            out[pre + "n_traj"] = np.array([len(traj_infos)])
            out[pre + "traj_lengths"] = np.array(sorted(int(t["Length"]) for t in traj_infos), dtype=np.int64)
        sampler.shutdown()
    _save("collector", out)


def gen_live_reference():
    """The reference's outputs on the seeded random cases of tests/live_reference_cases.py: returns, PPO loss,
    DQN loss (with gradients) and sum-tree op sequences."""
    from collections import namedtuple
    import torch
    sys.path.insert(0, os.path.dirname(HERE))                     # tests/
    import live_reference_cases as C
    from rlpyt.agents.base import AgentInputs
    from rlpyt.algos import utils as R
    from rlpyt.algos.dqn.dqn import DQN
    from rlpyt.algos.pg.ppo import PPO
    from rlpyt.distributions.categorical import Categorical, DistInfo
    from rlpyt.replays.sum_tree import SumTree
    out = {}
    for seed in C.RETURNS_SEEDS:
        c, pre = C.returns_case(seed), f"returns/{seed}/"
        done_f = c["done"].astype(np.float32)
        out[pre + "adv"], out[pre + "ret"] = R.generalized_advantage_estimation(c["reward"], c["value"], done_f, c["bv"],
                                                                              c["gamma"], c["lam"])
        out[pre + "discount_return"] = R.discount_return(c["reward"], done_f, c["bv"], c["gamma"])
        out[pre + "valid"] = R.valid_from_done(torch.from_numpy(done_f)).numpy()
        nstep = [R.discount_return_n_step(c["reward"], c["done"], n, c["gamma"], do_truncated=trunc)
                 for n, trunc in c["n_steps"]]
        out[pre + "nstep_shape"] = np.array([r.shape for r, _ in nstep], np.int64)   # truncated returns are shorter
        out[pre + "nstep_return"] = np.concatenate([r.ravel() for r, _ in nstep])
        out[pre + "nstep_done"] = np.concatenate([d.ravel() for _, d in nstep])

    class PgStub:
        recurrent = False

        def __init__(self, p, v, dist):
            self.p, self.v, self.distribution = p, v, dist

        def __call__(self, observation, prev_action, prev_reward):
            return DistInfo(prob=self.p), self.v

    for seed in C.PG_SEEDS:
        c, pre = C.pg_case(seed), f"pg/{seed}/"
        N, A = c["p_new"].shape
        p = torch.from_numpy(c["p_new"]).clone().requires_grad_(True)
        v = torch.from_numpy(c["value"]).clone().requires_grad_(True)
        algo = PPO(value_loss_coeff=c["c_v"], entropy_loss_coeff=c["c_ent"], ratio_clip=c["clip"])
        algo.agent = PgStub(p, v, Categorical(dim=A))
        z = torch.zeros(N)
        loss, ent, perp = algo.loss(AgentInputs(z, z, z), torch.from_numpy(c["action"]), torch.from_numpy(c["ret"]),
                                    torch.from_numpy(c["adv"]), None if c["valid"] is None else torch.from_numpy(c["valid"]),
                                    DistInfo(prob=torch.from_numpy(c["p_old"])))
        loss.backward()
        out[pre + "loss_entropy_perplexity"] = np.array([loss.item(), ent.item(), perp.item()], np.float64)
        out[pre + "grad_prob"], out[pre + "grad_value"] = p.grad.numpy(), v.grad.numpy()

    S = namedtuple("S", "agent_inputs action return_ done done_n target_inputs is_weights")
    for seed in C.DQN_SEEDS:
        c, pre = C.dqn_case(seed), f"dqn/{seed}/"
        N = len(c["action"])
        q = torch.from_numpy(c["qs"]).clone().requires_grad_(True)

        class Stub:
            def __call__(self, observation, prev_action, prev_reward):
                return q if int(observation[0]) == 0 else torch.from_numpy(c["nq"])

            def target(self, observation, prev_action, prev_reward):
                return torch.from_numpy(c["tq"])

        algo = DQN(discount=c["discount"], delta_clip=c["clip"], n_step_return=c["n_step"], double_dqn=c["double"],
                   prioritized_replay=c["pri"])
        algo.mid_batch_reset, algo.agent = True, Stub()
        z = torch.zeros(N)
        loss, td = algo.loss(S(AgentInputs(z, z, z), torch.from_numpy(c["action"]), torch.from_numpy(c["ret"]),
                               torch.from_numpy(c["done_n"]), torch.from_numpy(c["done_n"]), AgentInputs(z + 1, z, z),
                               torch.from_numpy(c["isw"])))
        loss.backward()
        out[pre + "loss"] = np.array([loss.item()], np.float64)
        out[pre + "td_abs_errors"], out[pre + "grad_qs"] = td.numpy(), q.grad.numpy()

    for seed in C.SUM_TREE_SEEDS:
        for k, x in C.sum_tree_trace(SumTree, seed).items():
            out[f"sum_tree/{seed}/{k}"] = x
    _save("live_reference", out)


GROUPS = {"returns": gen_returns, "loss": gen_loss, "ppo": gen_ppo, "replay": gen_replay, "dqn": gen_dqn,
          "collector": gen_collector, "ppo_lstm": gen_ppo_lstm, "seq_replay": gen_seq_replay, "r2d1": gen_r2d1,
          "live_reference": gen_live_reference}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    _import_reference()
    only = [s for s in args.only.split(",") if s]
    for name, fn in GROUPS.items():
        if only and name not in only:
            continue
        fn()


if __name__ == "__main__":
    main()
