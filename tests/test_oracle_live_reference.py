"""Property tests of the oracle against the UNMODIFIED reference on random shapes / seeds beyond the golden
cases (tests/live_reference_cases.py; the reference's outputs are stored in tests/golden/live_reference.npz by
``tests/golden/make_golden.py --only live_reference``): returns (bit-exact), PPO / A2C / DQN losses with
gradients (bit-exact, same torch ops), sum-tree op sequences (bit-exact tree contents and samples)."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import live_reference_cases as C  # noqa: E402


@pytest.fixture(scope="module")
def ref(golden):
    return golden("live_reference")


@pytest.mark.parametrize("seed", C.RETURNS_SEEDS)
def test_returns_random_shapes(ref, seed):
    from oracle import returns as O
    c, pre = C.returns_case(seed), f"returns/{seed}/"
    reward, value, done, bv, gam, lam = c["reward"], c["value"], c["done"], c["bv"], c["gamma"], c["lam"]
    o_adv, o_ret = O.generalized_advantage_estimation(reward, value, done, bv, gam, lam)
    assert np.array_equal(ref[pre + "adv"], o_adv) and np.array_equal(ref[pre + "ret"], o_ret)
    assert np.array_equal(ref[pre + "discount_return"], O.discount_return(reward, done, bv, gam))
    assert np.array_equal(ref[pre + "valid"], O.valid_from_done(done))
    nstep = [O.discount_return_n_step(reward, done, n, gam, do_truncated=trunc) for n, trunc in c["n_steps"]]
    assert np.array_equal(ref[pre + "nstep_shape"], [r.shape for r, _ in nstep])
    assert np.array_equal(ref[pre + "nstep_shape"], [d.shape for _, d in nstep])
    assert np.array_equal(ref[pre + "nstep_return"], np.concatenate([r.ravel() for r, _ in nstep]))
    assert np.array_equal(ref[pre + "nstep_done"], np.concatenate([d.ravel() for _, d in nstep]))


@pytest.mark.parametrize("seed", C.PG_SEEDS)
def test_pg_losses_random(ref, seed):
    from oracle import pg_loss as L
    c, pre = C.pg_case(seed), f"pg/{seed}/"
    o = L.ppo_loss(c["p_new"], c["value"], c["p_old"], c["action"], c["ret"], c["adv"], c["valid"], c["clip"], c["c_v"],
                   c["c_ent"])
    assert [o["loss"], o["entropy"], o["perplexity"]] == ref[pre + "loss_entropy_perplexity"].tolist()
    assert np.array_equal(o["grad_prob"], ref[pre + "grad_prob"]) and np.array_equal(o["grad_value"], ref[pre + "grad_value"])


@pytest.mark.parametrize("seed", C.DQN_SEEDS)
def test_dqn_loss_random(ref, seed):
    from oracle.dqn_loss import dqn_loss
    c, pre = C.dqn_case(seed), f"dqn/{seed}/"
    t = torch.from_numpy
    o_loss, o_td, o_grad = dqn_loss(t(c["qs"]), t(c["tq"]), t(c["nq"]) if c["double"] else None, t(c["action"]), t(c["ret"]),
                                    t(c["done_n"]), t(c["isw"]) if c["pri"] else None, c["discount"], c["n_step"], c["clip"])
    assert float(o_loss) == float(ref[pre + "loss"][0])
    assert np.array_equal(o_td.numpy(), ref[pre + "td_abs_errors"]) and np.array_equal(o_grad.numpy(), ref[pre + "grad_qs"])


@pytest.mark.parametrize("seed", C.SUM_TREE_SEEDS)
def test_sum_tree_random_op_sequences(ref, seed):
    from oracle.sum_tree import SumTree
    got = C.sum_tree_trace(SumTree, seed)
    for k, x in got.items():
        want = ref[f"sum_tree/{seed}/{k}"]
        assert x.shape == want.shape and np.array_equal(x, want), k
