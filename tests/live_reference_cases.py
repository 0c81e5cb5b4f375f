"""Seeded random cases of tests/test_oracle_live_reference.py: random shapes and hyper-parameters beyond the
fixed golden cases.  ``tests/golden/make_golden.py --only live_reference`` runs the unmodified reference on them
and stores its outputs in tests/golden/live_reference.npz; the test runs the oracle on the same cases."""
import numpy as np

RETURNS_SEEDS, PG_SEEDS, DQN_SEEDS, SUM_TREE_SEEDS = range(8), range(6), range(6), range(5)


def returns_case(seed):
    rng = np.random.default_rng(100 + seed)
    T, B = int(rng.integers(1, 40)), int(rng.integers(1, 9))
    reward = rng.standard_normal((T, B)).astype(np.float32)
    value = rng.standard_normal((T, B)).astype(np.float32)
    done = rng.random((T, B)) < 0.15
    bv = rng.standard_normal((1, B)).astype(np.float32)
    gamma, lam = float(rng.choice([0.99, 0.9, 1.0, 0.5])), float(rng.choice([1.0, 0.98, 0.95, 0.0]))
    n_steps = [(n, trunc) for n in range(1, min(T, 5) + 1) for trunc in (False, True)]
    return dict(reward=reward, value=value, done=done, bv=bv, gamma=gamma, lam=lam, n_steps=n_steps)


def pg_case(seed):
    rng = np.random.default_rng(200 + seed)
    N, A = int(rng.integers(1, 300)), int(rng.integers(2, 19))
    p_new = rng.dirichlet(np.ones(A), N).astype(np.float32)
    p_old = rng.dirichlet(np.ones(A), N).astype(np.float32)
    value, ret, adv = (rng.standard_normal(N).astype(np.float32) for _ in range(3))
    action = rng.integers(0, A, N).astype(np.int64)
    valid = (rng.random(N) < 0.8).astype(np.float32) if seed % 2 else None
    if valid is not None:
        valid[0] = 1.0
    return dict(p_new=p_new, p_old=p_old, value=value, ret=ret, adv=adv, action=action, valid=valid,
                clip=0.1 + 0.1 * (seed % 3), c_v=0.5 + 0.25 * seed, c_ent=0.01 * seed)


def dqn_case(seed):
    rng = np.random.default_rng(300 + seed)
    N, A = int(rng.integers(1, 200)), int(rng.integers(2, 19))
    qs, tq, nq = ((rng.standard_normal((N, A)) * 2).astype(np.float32) for _ in range(3))
    action = rng.integers(0, A, N).astype(np.int64)
    ret = rng.standard_normal(N).astype(np.float32)
    done_n = rng.random(N) < 0.2
    isw = (rng.random(N) * 0.9 + 0.1).astype(np.float32)
    return dict(qs=qs, tq=tq, nq=nq, action=action, ret=ret, done_n=done_n, isw=isw,
                double=bool(seed & 1), pri=bool(seed & 2), clip=[1.0, None, 0.25][seed % 3],
                n_step=1 + seed % 4, discount=[0.99, 0.9][seed % 2])


def sum_tree_trace(tree_cls, seed):
    """Drive a sum tree (the reference's class or the oracle's: same constructor and methods) through a seeded
    sequence of advance / sample / update_batch_priorities.  Returns ``trees``: the whole tree after every
    advance and every update, in order; ``T_idxs`` / ``B_idxs`` / ``priorities``: every sample drawn, concatenated;
    ``n_sampled``: the length of each draw.  Sampling draws from the global numpy stream, like the reference."""
    rng = np.random.default_rng(400 + seed)
    T, B = int(rng.integers(12, 40)), int(rng.integers(1, 6))
    off_b, off_f = int(rng.integers(1, 4)), int(rng.integers(1, 4))
    dv = float(rng.choice([1.0, 0.5, 2.0]))
    tree = tree_cls(T, B, off_b, off_f, default_value=dv)
    trees, samples = [], []
    for step in range(30):
        adv = int(rng.integers(1, 5))
        tree.advance(adv)
        trees.append(tree.tree.copy())
        if tree.tree[0] <= 0:
            continue
        n = int(rng.integers(1, 9))
        unique = bool(step % 3 == 0) and 2 * n <= int((tree.priorities > 0).sum())
        np.random.seed(1000 * seed + step)
        (t_idxs, b_idxs), pri_sampled = tree.sample(n, unique=unique)
        samples.append((t_idxs, b_idxs, pri_sampled))
        pri = (rng.random(len(t_idxs)) + 0.01).astype(np.float32)
        tree.update_batch_priorities(pri)
        trees.append(tree.tree.copy())
    return dict(trees=np.stack(trees), T_idxs=np.concatenate([s[0] for s in samples]),
                B_idxs=np.concatenate([s[1] for s in samples]), priorities=np.concatenate([s[2] for s in samples]),
                n_sampled=np.array([len(s[0]) for s in samples], np.int64))
