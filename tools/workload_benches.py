"""bench.py --workload gae | replay | dqn: BASELINE.json configs[1] and configs[3] in the same line format as the
PPO workload (metric/value/unit, e2e through the public API with HOST buffers, roofline of the dominant kernel
against MEASURED_PEAKS.json, cpu_baseline = the unmodified reference from oracle/_ref on the host cores, or
the oracle port when it is absent).  The driver only runs the default PPO workload; lines of these workloads
measured on a B200 are kept under profiles/ (tools/run_workloads.sh).

    python bench.py --workload gae    [--steps 50 --warmup 5]
    python bench.py --workload replay [--steps 200 --warmup 10]
    python bench.py --workload dqn    [--steps 200 --warmup 5]
"""
import json
import os
import sys
import time
from collections import namedtuple

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md)"


def _events(fn, reps, flush=None):
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    return float(np.mean(ts))


def _ref_import():
    from baseline import reference_arm as R
    if not R.available():
        return False
    R._import()
    return True


def _clocks(local_rank=0):
    sys.path.insert(0, ROOT)
    from bench import ClockSampler
    return ClockSampler(local_rank)


def _line(metric, unit, value, ms, K, W, workload, extra):
    out = {"metric": metric, "value": value, "unit": unit, "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic",
           "config": {"workload": workload}}
    out.update(extra)
    return out


# ------------------------------------------------------------------------------------------------ gae
def run_gae(args):
    """configs[1]: GAE / discount-return kernel vs numpy on synthetic [T=128,B=256] fp32 - and the metric's
    "GAE-scan GB/s" at the HBM-bound size [128, 2^20] (inputs 2.3 GB, far larger than L2)."""
    from rlpyt_b200 import _lib
    from rlpyt_b200.algos import utils as U
    _lib.load()
    K, W = max(args.steps, 10), max(args.warmup, 3)
    peak, how = _peak()
    T, Bs, Bl = 128, 256, 1 << 20
    gen = torch.Generator(device="cuda").manual_seed(0)

    def dev_case(B):
        r = torch.randn(T, B, device="cuda", generator=gen)
        v = torch.randn(T, B, device="cuda", generator=gen)
        d = torch.rand(T, B, device="cuda", generator=gen) < 0.01
        b = torch.randn(1, B, device="cuda", generator=gen)
        return r, v, d, b, torch.empty_like(r), torch.empty_like(r)
    r, v, d, b, adv, ret = dev_case(Bl)
    big = lambda: U.generalized_advantage_estimation(r, v, d, b, 0.99, 0.98, advantage_dest=adv, return_dest=ret, algo=1)
    for _ in range(W):
        big()
    torch.cuda.synchronize()
    l0 = _lib.launch_count
    with _clocks() as clk:
        t_big = _events(big, K)
    launches = _lib.launch_count - l0
    nbytes = T * Bl * 17 + 4 * Bl
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))["gae_stream_bytes_per_launch"]
    except Exception:  # noqa: BLE001
        pass
    rs, vs, ds, bs, advs, rets = dev_case(Bs)
    lat = {}
    for name, algo in (("tscan", 2), ("stream", 1)):
        fn = lambda: U.generalized_advantage_estimation(rs, vs, ds, bs, 0.99, 0.98, advantage_dest=advs, return_dest=rets, algo=algo)
        for _ in range(W):
            fn()
        torch.cuda.synchronize()
        # device time of ONE launch: 20 launches captured back to back in a CUDA graph (an isolated launch from Python
        # is timed together with ~20 us of launch latency on an idle GPU)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(20):
                fn()
        graph.replay()
        lat[name] = _events(graph.replay, K) * 1e6 / 20
        lat[name + "_single_call_from_python"] = _events(fn, K) * 1e6
    # e2e: the public function with HOST (numpy) arrays at the config's size: H2D + kernel + D2H inside the clock
    rng = np.random.default_rng(0)
    hr, hv = rng.standard_normal((T, Bs)).astype(np.float32), rng.standard_normal((T, Bs)).astype(np.float32)
    hd, hb = rng.random((T, Bs)) < 0.01, rng.standard_normal((1, Bs)).astype(np.float32)
    pin = lambda a: torch.from_numpy(a).pin_memory()
    pr, pv, pd, pb = pin(hr), pin(hv), pin(hd), pin(hb)
    out_a, out_r = torch.empty(T, Bs).pin_memory(), torch.empty(T, Bs).pin_memory()

    def host_call():
        a, rr = U.generalized_advantage_estimation(pr.cuda(non_blocking=True), pv.cuda(non_blocking=True), pd.cuda(non_blocking=True),
                                                   pb.cuda(non_blocking=True), 0.99, 0.98)
        out_a.copy_(a, non_blocking=True)
        out_r.copy_(rr, non_blocking=True)
        torch.cuda.synchronize()
    for _ in range(W):
        host_call()
    t0 = time.perf_counter()
    for _ in range(K):
        host_call()
    t_host = (time.perf_counter() - t0) / K
    small_bytes = T * Bs * 17 + 4 * Bs
    # CPU: the reference's own function (torch-CPU path = what PPO runs; numpy path), same [128,256] inputs
    kind = "port"
    if _ref_import():
        from rlpyt.algos.utils import generalized_advantage_estimation as ref_gae
        kind = "reference"
    else:
        from oracle.returns import generalized_advantage_estimation as ref_gae
    tr, tv, td, tb = (torch.from_numpy(x) for x in (hr, hv, hd.astype(np.float32), hb))
    for _ in range(3):
        ref_gae(tr, tv, td, tb, 0.99, 0.98)
    reps = 50
    t0 = time.perf_counter()
    for _ in range(reps):
        ref_gae(tr, tv, td, tb, 0.99, 0.98)
    cpu_torch = (time.perf_counter() - t0) / reps
    t0 = time.perf_counter()
    for _ in range(reps):
        ref_gae(hr, hv, hd, hb, 0.99, 0.98)
    cpu_np = (time.perf_counter() - t0) / reps
    out = _line("GAE-scan GB/s (GAE / discount-return kernel, fp32)", "GB/s", nbytes / t_big / 1e9, t_big * 1e3, K, W,
                "GAE scan gamma .99 lambda .98: [T=128,B=2^20] for the HBM-bound GB/s (BASELINE.json configs[1] is [128,256]: "
                "see latency_us)", {
        "dtype": "f32", "gpu_launches": launches, "clocks": clk.summary(),
        "config_l2": "inputs_larger_than_L2 (2.3 GB per launch)",
        "latency_us_128x256": {"returns_tscan_kernel": lat["tscan"], "returns_stream_kernel": lat["stream"],
                               "tscan_single_call_from_python": lat["tscan_single_call_from_python"],
                               "algorithmic_bytes": small_bytes},
        "e2e": {"value": small_bytes / t_host / 1e9, "unit": "GB/s", "us_per_call": t_host * 1e6,
                "what": "generalized_advantage_estimation on pinned HOST arrays [128,256]: H2D + kernel + D2H, wall clock",
                "h2d_bytes_per_step": T * Bs * 9 + 4 * Bs, "d2h_bytes_per_step": T * Bs * 8},
        "roofline": {"kernel": "returns_stream_kernel<4,GAE> [T=128, B=2^20]", "bound": "hbm", "achieved": nbytes / t_big / 1e9,
                     "peak": peak, "unit": "GB/s", "frac": nbytes / t_big / 1e9 / peak, "traffic": traffic,
                     "peak_source": how, "us_per_launch": t_big * 1e6, "algorithmic_bytes": nbytes},
        "cpu_baseline": {"value": small_bytes / cpu_torch / 1e9, "unit": "GB/s", "cores": torch.get_num_threads(), "kind": kind,
                         "sample": f"rlpyt.algos.utils.generalized_advantage_estimation on torch-CPU tensors [128,256] (what PPO "
                                   f"runs), {reps} calls", "us_per_call_torch_cpu": cpu_torch * 1e6,
                         "us_per_call_numpy": cpu_np * 1e6,
                         "speedup_kernel_vs_torch_cpu": cpu_torch * 1e6 / lat["tscan"]},
    })
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------ replay
def _fill_replay(size, B=256):
    from rlpyt_b200.replays.non_sequence.frame import PrioritizedReplayFrameBuffer
    from rlpyt_b200.utils.collections import namedarraytuple
    Ex = namedarraytuple("SamplesToBuffer", ["observation", "action", "reward", "done"])
    ex = Ex(observation=np.zeros((4, 84, 84), np.uint8), action=np.int64(0), reward=np.float32(0), done=np.bool_(False))
    buf = PrioritizedReplayFrameBuffer(example=ex, size=size, B=B, discount=0.99, n_step_return=3, alpha=0.6, beta=0.4,
                                       default_priority=1)
    T = 128
    g = torch.Generator(device="cuda").manual_seed(0)
    obs = torch.randint(0, 256, (T, B, 4, 84, 84), dtype=torch.uint8, device="cuda", generator=g)
    for _ in range(buf.T // T + 2):
        buf.append_samples(Ex(observation=obs, action=torch.randint(0, 6, (T, B), device="cuda", generator=g),
                              reward=torch.randn(T, B, device="cuda", generator=g),
                              done=torch.rand(T, B, device="cuda", generator=g) < 0.005))
    return buf


def _cpu_replay(n_frames, reps):
    """sample_batch(512) / update_batch_priorities(512) of the reference's PrioritizedReplayFrameBuffer on the host
    (bounded: a 100 K-frame ring - per-batch cost depends on the ring size only through the tree depth)."""
    rng = np.random.default_rng(0)
    T, B = 64, 256
    obs = rng.integers(0, 256, size=(T, B, 4, 84, 84), dtype=np.uint8)
    if _ref_import():
        from rlpyt.replays.non_sequence.frame import PrioritizedReplayFrameBuffer as RefBuf
        from rlpyt.utils.collections import namedarraytuple as ref_nat
        Ex = ref_nat("SamplesToBuffer", ["observation", "action", "reward", "done"])
        ex = Ex(observation=np.zeros((4, 84, 84), np.uint8), action=np.int64(0), reward=np.float32(0), done=np.bool_(False))
        o = RefBuf(example=ex, size=n_frames, B=B, discount=0.99, n_step_return=3, alpha=0.6, beta=0.4, default_priority=1)
        for _ in range(n_frames // (T * B) + 2):
            o.append_samples(Ex(observation=torch.from_numpy(obs), action=torch.from_numpy(rng.integers(0, 6, (T, B))),
                                reward=torch.from_numpy(rng.standard_normal((T, B)).astype(np.float32)),
                                done=torch.from_numpy(rng.random((T, B)) < 0.005)))
        new = torch.from_numpy(np.abs(rng.standard_normal(512)).astype(np.float32))
        kind = "reference"
    else:
        from oracle.replay import FrameReplay
        o = FrameReplay((4, 84, 84), n_frames, B, discount=0.99, n_step_return=3)
        for _ in range(n_frames // (T * B) + 2):
            o.append_samples(dict(observation=obs, action=rng.integers(0, 6, (T, B)),
                                  reward=rng.standard_normal((T, B)).astype(np.float32), done=rng.random((T, B)) < 0.005))
        new = np.abs(rng.standard_normal(512)).astype(np.float32)
        kind = "port"
    o.sample_batch(512)
    t_s = t_u = 0.0
    for _ in range(reps):
        t0 = time.perf_counter()
        o.sample_batch(512)
        t1 = time.perf_counter()
        o.update_batch_priorities(new)
        t_u += time.perf_counter() - t1
        t_s += t1 - t0
    return t_s / reps, t_u / reps, kind


def run_replay(args):
    """configs[3]: prioritized frame replay, 1 M-frame buffer, batch 512, n-step 3: sum-tree sample + frame gather +
    priority update.  step = sample_batch(512) + update_batch_priorities(512)."""
    from rlpyt_b200 import _lib
    _lib.load()
    K, W = max(args.steps, 20), max(args.warmup, 3)
    peak, how = _peak()
    buf = _fill_replay(1_000_000)
    np.random.seed(0)
    pri = torch.rand(512, device="cuda") + 0.01

    def step():
        buf.sample_batch(512)
        buf.update_batch_priorities(pri)
    for _ in range(W):
        step()
    torch.cuda.synchronize()
    l0 = _lib.launch_count
    with _clocks() as clk:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            step()
        e1.record()
        torch.cuda.synchronize()
    dt = e0.elapsed_time(e1) * 1e-3 / K
    launches = _lib.launch_count - l0
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    t_sample = _events(lambda: buf.sample_batch(512), 20, flush)
    buf.sample_batch(512)
    t_update = _events(lambda: buf.update_batch_priorities(pri), 20)
    (T_idxs, B_idxs), _p = buf.priority_tree.sample(512)
    t_ext = _events(lambda: buf.extract_batch(T_idxs, B_idxs), 20, flush)
    nbytes = 2 * 2 * 512 * 4 * 84 * 84
    # the same kernel on a batch large enough to amortise launch + the per-CTA latency chain (index -> done flags ->
    # frames -> store): what the data movement itself sustains
    n_big = 8192
    (T_big, B_big), _p = buf.priority_tree.sample(n_big)
    t_big = _events(lambda: buf.extract_batch(T_big, B_big), 10, flush)
    nbytes_big = 2 * 2 * n_big * 4 * 84 * 84
    # e2e: the batch lands in pinned host memory, the new priorities come from the host
    host_pri = (torch.rand(512) + 0.01).pin_memory()
    b0 = buf.sample_batch(512)
    host_obs = torch.empty_like(b0.agent_inputs.observation, device="cpu").pin_memory()
    host_tgt = torch.empty_like(b0.target_inputs.observation, device="cpu").pin_memory()

    def host_step():
        b = buf.sample_batch(512)
        host_obs.copy_(b.agent_inputs.observation, non_blocking=True)
        host_tgt.copy_(b.target_inputs.observation, non_blocking=True)
        buf.update_batch_priorities(host_pri.cuda(non_blocking=True))
        torch.cuda.synchronize()
    for _ in range(W):
        host_step()
    t0 = time.perf_counter()
    for _ in range(K):
        host_step()
    t_host = (time.perf_counter() - t0) / K
    cpu_s, cpu_u, kind = _cpu_replay(100_000, 20)
    out = _line("prioritized frame-replay transitions/s (sample_batch(512) + update_batch_priorities, 1M frames, n-step 3)",
                "transitions/s", 512 / dt, dt * 1e3, K, W,
                f"PrioritizedReplayFrameBuffer {buf.size} frames x (84,84) u8 (7 GB in HBM), B=256, batch 512, n-step 3, "
                "alpha .6 beta .4 (BASELINE.json configs[3])", {
        "dtype": "u8 frames, f64 sum-tree, int64 indices", "gpu_launches": launches, "clocks": clk.summary(),
        "config_l2": "replay store (7 GB) larger than L2; flushed between the per-phase timings",
        "phases_us": {"sample_batch": t_sample * 1e6, "update_batch_priorities": t_update * 1e6, "replay_extract_bulk_kernel": t_ext * 1e6},
        "e2e": {"value": 512 / t_host, "unit": "transitions/s", "us_per_step": t_host * 1e6,
                "what": "sample_batch -> observations copied to pinned host memory; priorities uploaded from the host",
                "h2d_bytes_per_step": 512 * 4, "d2h_bytes_per_step": 2 * 512 * 4 * 84 * 84},
        "roofline": {"kernel": "replay_extract_bulk_kernel (512 samples x 2 stacks of 4 frames, cp.async.bulk)", "bound": "hbm", "achieved": nbytes / t_ext / 1e9,
                     "peak": peak, "unit": "GB/s", "frac": nbytes / t_ext / 1e9 / peak, "traffic": None, "peak_source": how,
                     "us_per_launch": t_ext * 1e6, "algorithmic_bytes": nbytes,
                     "at_batch_8192": {"us_per_launch": t_big * 1e6, "achieved": nbytes_big / t_big / 1e9,
                                       "frac": nbytes_big / t_big / 1e9 / peak, "algorithmic_bytes": nbytes_big,
                                       "note": "batch 512 moves 58 MB in one wave of 1024 CTAs: launch + one latency chain "
                                               "(index -> done flags -> frames -> store, ~4 us) bound it near 0.6 of peak; 16x the "
                                               "batch shows the kernel's own bandwidth"}},
        "cpu_baseline": {"value": 512 / (cpu_s + cpu_u), "unit": "transitions/s", "cores": 1, "kind": kind,
                         "sample": "PrioritizedReplayFrameBuffer.sample_batch(512) + update_batch_priorities on the host, "
                                   "100 K-frame ring, 20 batches", "sample_batch_us": cpu_s * 1e6, "update_us": cpu_u * 1e6},
    })
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------ dqn
def run_dqn(args):
    """configs[3] end to end (SURVEY 8(f) row 1): one DQN update = sample_batch(512) -> online/target forwards ->
    fused loss -> backward -> clip+Adam -> priority update, replay resident in HBM."""
    from tools import bench_dqn as BD
    from rlpyt_b200 import _lib
    from rlpyt_b200.agents.dqn.atari.atari_dqn_agent import AtariDqnAgent
    from rlpyt_b200.algos.dqn.dqn import DQN
    from rlpyt_b200.samplers.collections import BatchSpec
    K, W = max(args.steps, 20), max(args.warmup, 3)
    peak, how = _peak()
    torch.manual_seed(0)
    np.random.seed(0)
    Spaces = namedtuple("Spaces", "observation action")
    agent = AtariDqnAgent()
    agent.initialize(Spaces(namedtuple("O", "shape")(BD.IMG), namedtuple("Ac", "n")(BD.A)))
    agent.to_device(0)
    algo = DQN(batch_size=512, min_steps_learn=0, replay_size=1_000_000, replay_ratio=8, n_step_return=3, double_dqn=True,
               prioritized_replay=True, target_update_interval=312)
    examples = dict(observation=np.zeros(BD.IMG, np.uint8), action=np.int64(0), reward=np.float32(0), done=np.bool_(False))
    algo.initialize(agent, n_itr=10 ** 6, batch_spec=BatchSpec(BD.T, BD.B), mid_batch_reset=True, examples=examples)
    buf = algo.replay_buffer
    data = [BD.synth(s, "cuda") for s in range(2)]
    for i in range(buf.T // BD.T + 2):
        buf.append_samples(algo.samples_to_buffer(data[i % 2]))
    agent.train_mode(0)
    host_loss = torch.empty(1).pin_memory()

    def update(read_back=False):
        batch = buf.sample_batch(512)
        algo.optimizer.zero_grad()
        loss, td = algo.loss(batch)
        loss.backward()
        algo.optimizer.clip_and_step(algo.clip_grad_norm)
        buf.update_batch_priorities(td)
        if read_back:
            host_loss.copy_(loss.detach().reshape(1), non_blocking=True)
            torch.cuda.synchronize()
    for _ in range(W):
        update()
    torch.cuda.synchronize()
    l0 = _lib.launch_count
    with _clocks() as clk:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            update()
        e1.record()
        torch.cuda.synchronize()
    dt = e0.elapsed_time(e1) * 1e-3 / K
    launches = _lib.launch_count - l0
    # e2e: one sampler batch [T=128? no - T=4,B=256 as replay_ratio 8 dictates] arrives from pinned HOST memory every 4 updates
    Th = 4
    host = BD.synth(7, "cpu") if hasattr(BD, "synth") else None
    host_obs = host.env.observation[:Th].pin_memory()

    def e2e_iter():
        s = data[0]
        s.env.observation[:Th].copy_(host_obs, non_blocking=True)      # H2D of the new frames
        for _ in range(1):
            update(read_back=True)
    for _ in range(W):
        e2e_iter()
    t0 = time.perf_counter()
    for _ in range(K):
        e2e_iter()
    t_host = (time.perf_counter() - t0) / K
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    (T_idxs, B_idxs), _p = buf.priority_tree.sample(512)
    t_ext = _events(lambda: buf.extract_batch(T_idxs, B_idxs), 20, flush)
    nbytes = 2 * 2 * 512 * 4 * 84 * 84
    a = namedtuple("A", "batch cpu_updates")(512, 3)
    cpu = BD.cpu_baseline(agent, a)
    out = _line("DQN updates/s (prioritized frame replay 1M frames, Double-DQN, n-step 3, batch 512)", "updates/s", 1.0 / dt,
                dt * 1e3, K, W, "AtariDqnAgent A=6 + DQN(double, prioritized, n-step 3) on a 1M-frame HBM replay, batch 512 "
                                "(BASELINE.json configs[3] + SURVEY 8(f) row 1)", {
        "dtype": "f32 network, u8 frames, f64 sum-tree", "gpu_launches": launches, "clocks": clk.summary(),
        "transitions_per_s": 512 / dt, "config_l2": "replay store (7 GB) larger than L2",
        "e2e": {"value": 1.0 / t_host, "unit": "updates/s", "what": "update + H2D of 4x256 new frames from pinned host memory + "
                "D2H of the loss, wall clock", "h2d_bytes_per_step": int(host_obs.numel()), "d2h_bytes_per_step": 4},
        "roofline": {"kernel": "replay_extract_bulk_kernel (512 samples x 2 stacks of 4 frames, cp.async.bulk)", "bound": "hbm", "achieved": nbytes / t_ext / 1e9,
                     "peak": peak, "unit": "GB/s", "frac": nbytes / t_ext / 1e9 / peak, "traffic": None, "peak_source": how,
                     "us_per_launch": t_ext * 1e6, "algorithmic_bytes": nbytes,
                     "note": "the update itself is dominated by the Q-network (forward x3 + backward at batch 512)"},
        "cpu_baseline": cpu,
    })
    print(json.dumps(out), flush=True)


def run(args):
    if args.impl == "reference":
        print(json.dumps({"impl": "reference", "unavailable": f"--workload {args.workload}: the reference's CPU timing is the "
                                                              "cpu_baseline object of the b200 line"}), flush=True)
        return
    {"gae": run_gae, "replay": run_replay, "dqn": run_dqn}[args.workload](args)
