#!/usr/bin/env python
"""bench.py - the driver's measurement contract.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload ppo|gae|replay|dqn]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

``--workload ppo`` (default) is the driver's contract, BASELINE.json configs[2] (configs[4] at N > 1); ``gae``
(configs[1]), ``replay`` and ``dqn`` (configs[3]) print the same kind of line for the other configurations
(tools/workload_benches.py; outputs of a B200 run are kept under profiles/).

Metric (BASELINE.json): env-steps/sec of PPO on Atari-shaped data, [T=128, B=256] per GPU, AtariFf
agent, the reference's PPO hyper-parameters (rlpyt/experiments/configs/atari/pg/atari_ff_ppo.py:5-16);
plus the GAE-scan GB/s in ``roofline``.

A "step" is one PPO iteration over one [T,B] batch of synthetic samples:
  value  - LEARNER ONLY: ``algo.optimize_agent`` on a batch already resident in HBM (returns + 4x4 minibatch
           updates: gather, forward, fused loss, backward, all-reduce, clip+Adam).  Compare it with the
           reference line's ``value`` (its optimize_agent alone), never with a loop that also samples;
  e2e    - the public API loop a user runs: ``sampler.obtain_samples`` (CPU synthetic envs in
           worker processes, per-step H2D of observations from pinned host memory, agent.step on
           the GPU, D2H of actions) followed by ``algo.optimize_agent`` (D2H of the OptInfo rows).
           This is the metric's number (env-steps/s of PPO); compare it with the reference line's ``e2e``.
Weak scaling: every rank owns B=256 environments; ``value``/``e2e`` are whole-job aggregates.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

T_CFG, B_CFG, IMAGE, N_ACTIONS = 128, 256, (4, 84, 84), 6
PPO_KW = dict(discount=0.99, learning_rate=1e-3, value_loss_coeff=1., entropy_loss_coeff=0.01,
              clip_grad_norm=1., gae_lambda=0.98, linear_lr_schedule=True, minibatches=4, epochs=4,
              ratio_clip=0.1)
ENV_KW = dict(image_shape=IMAGE, n_actions=N_ACTIONS, p_done=1 / 500., p_reward=0.04)


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self._stop = index, [], threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=3)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]),
                "power_w_max": max(float(r[2]) for r in self.rows), "reasons": reasons, "samples": len(self.rows)}


# --------------------------------------------------------------------------------------------- b200 arm
def run_b200(args):
    import torch.distributed as dist
    from rlpyt_b200 import _lib
    from rlpyt_b200.agents.pg.atari import AtariFfAgent
    from rlpyt_b200.algos.pg.ppo import PPO
    from rlpyt_b200.algos import utils as U
    from rlpyt_b200.envs.synthetic import SyntheticAtariEnv
    from rlpyt_b200.samplers.parallel.gpu.sampler import GpuSampler

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    all_cpus = sorted(os.sched_getaffinity(0))
    cores = len(all_cpus)
    seed = 0 + 100 * rank                                            # sync_rl.py:82 seeds per rank
    np.random.seed(seed)
    torch.manual_seed(seed)
    SamplerCls = GpuSampler
    sampler_kind = os.environ.get("RLPYT_B200_BENCH_SAMPLER", args.sampler)
    if sampler_kind == "alternating":   # two worker groups: one steps its envs while the GPU serves the other
        from rlpyt_b200.samplers.parallel.gpu.alternating_sampler import AlternatingSampler as SamplerCls
    sampler = SamplerCls(EnvCls=SyntheticAtariEnv, env_kwargs=ENV_KW, batch_T=T_CFG, batch_B=B_CFG,
                         max_decorrelation_steps=20)
    agent = AtariFfAgent()
    from rlpyt_b200.utils.affinity import make_affinity
    # every GPU gets the same host share at every N: one eighth of the box's PHYSICAL cores (an 8-GPU node),
    # the first of them for the master, one env worker per hardware thread of the others (--workers-per-core 1:
    # one per core).  Measured on the 2 x 64-thread host (profiles/r02_sampler_configs.txt): alternating + 14
    # workers on 7 cores hides the env stepping behind the device half-steps (59 ms per batch; standard 76-79 ms).
    affinity = make_affinity(local_rank, args.workers or None, local_rank=local_rank, ranks_per_node=world,
                             node_share=8, smt_workers=args.workers_per_core >= 2)
    if sampler_kind == "alternating" and len(affinity["workers_cpus"]) % 2:
        # two equal worker groups: drop the odd worker; a share with one worker core runs one worker per group on it
        wc = affinity["workers_cpus"]
        affinity["workers_cpus"] = wc[:-1] if len(wc) > 1 else wc * 2
    n_workers = len(affinity["workers_cpus"])
    sampler.initialize(agent, affinity=affinity, seed=seed + 1, bootstrap_value=True, world_size=world, rank=rank)
    agent.to_device(local_rank)
    if world > 1:
        agent.data_parallel()
    algo = PPO(**PPO_KW)
    n_itr = 10 ** 6
    algo.initialize(agent, n_itr, sampler.batch_spec, mid_batch_reset=sampler.mid_batch_reset,
                    world_size=world, rank=rank)
    steps_per_itr = T_CFG * B_CFG * world
    K, W = args.steps, args.warmup
    itr = 0
    try:
        # ---- batch resident in HBM
        samples, _ = sampler.obtain_samples(itr)
        agent.train_mode(itr)
        for _ in range(W):
            algo.optimize_agent(itr, samples)
            itr += 1
        barrier()
        l0 = _lib.launch_count
        with ClockSampler(local_rank) as clk_value:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(K):
                info = algo.optimize_agent(itr, samples)
                itr += 1
            e1.record()
            barrier()
        t_value = max_over_ranks(e0.elapsed_time(e1) * 1e-3)
        launches = _lib.launch_count - l0
        dumps = step_outputs("learner", info, agent) if args.dump_outputs else {}
        value = steps_per_itr * K / t_value
        # device time of the returns + loss kernels INSIDE a real optimize_agent iteration (CUDA events around
        # process_returns and around each fused-loss call; the stream is kept busy by the network kernels, so the
        # Python/ctypes cost of issuing them is hidden - unlike a stand-alone eager loop)
        algo.profile_events = []
        algo.optimize_agent(itr, samples)
        itr += 1
        torch.cuda.synchronize()
        evs = algo.profile_events
        algo.profile_events = None
        in_situ_ms = sum(evs[i].elapsed_time(evs[i + 1]) for i in range(0, len(evs) - 1, 2))

        # ---- end to end through the public API (host buffers, H2D/D2H inside the timed region)
        for _ in range(W):
            agent.sample_mode(itr)
            samples, _ = sampler.obtain_samples(itr)
            agent.train_mode(itr)
            algo.optimize_agent(itr, samples)
            itr += 1
        barrier()
        t_sample = 0.0
        if getattr(sampler, "profile", None):
            for k in sampler.profile:
                sampler.profile[k] = 0
        with ClockSampler(local_rank) as clk_e2e:
            t0 = time.perf_counter()
            for _ in range(K):
                agent.sample_mode(itr)
                ts = time.perf_counter()
                samples, traj_infos = sampler.obtain_samples(itr)
                t_sample += time.perf_counter() - ts
                agent.train_mode(itr)
                info = algo.optimize_agent(itr, samples)
                itr += 1
            barrier()
            t_e2e = max_over_ranks(time.perf_counter() - t0)
        if args.dump_outputs:
            dumps.update(step_outputs("e2e", info, agent, samples))
        e2e = steps_per_itr * K / t_e2e
        sampler_profile = None
        pr = getattr(sampler, "profile", None)
        if pr and pr.get("steps"):   # RLPYT_B200_SAMPLER_PROFILE=1: master-side split of one env step
            sampler_profile = {k[:-2]: pr[k] / pr["steps"] * 1e6 for k in pr if k.endswith("_s")}
            if "early_uploads" in pr:
                sampler_profile["early_upload_frac"] = pr["early_uploads"] / (2 * pr["steps"])
        params_identical = None
        if world > 1:   # data-parallel replicas must hold bit-identical parameters after K+W updates x 16
            flat = algo.optimizer.flat_param if hasattr(algo.optimizer, "flat_param") else torch.cat(
                [p.detach().reshape(-1) for p in agent.parameters()])
            mine = torch.stack([flat.double().sum(), flat.double().abs().sum(),
                                flat.view(torch.int32).long().sum().double()])
            allv = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(allv, mine)
            params_identical = bool(all(torch.equal(v, allv[0]) for v in allv))
        obs_bytes = int(np.prod(IMAGE))
        h2d = (T_CFG + 1) * B_CFG * (obs_bytes + 4 + 1) + 16 * (T_CFG * B_CFG // 4) * 8
        d2h = T_CFG * B_CFG * 8 + 16 * 4 * 4
    finally:
        sampler.shutdown()
        try:
            os.sched_setaffinity(0, all_cpus)  # the sampler pinned the master near its GPU; undo for the CPU legs
        except OSError:
            pass

    out = {
        "metric": "env-steps/sec PPO Atari [T=128,B=256] at 1/2/4/8 GPU; GAE-scan GB/s",
        "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": t_value / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "value_scope": "learner only: algo.optimize_agent on an HBM-resident [T,B] batch; the metric itself "
                       "(sampler + learner through the public API, host buffers) is e2e",
        "config": {"workload": "PPO+AtariFfAgent, synthetic Atari env obs (4,84,84) u8, T=128 B=256 per GPU "
                               "(BASELINE.json configs[2]; configs[4] at N>1), gamma .99 lambda .98 lr 1e-3 clip .1 4x4",
                   "global_batch": steps_per_itr, "parallelism": f"dp{world}",
                   "l2": "inputs_larger_than_L2 (925 MB observation batch per rank)",
                   "env_workers_per_rank": n_workers, "host_threads": cores, "sampler": sampler_kind,
                   "worker_cpus_rank0": [c[0] for c in affinity["workers_cpus"]], "master_cpus_rank0": affinity["master_cpus"]},
        "e2e": {"value": e2e, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": t_e2e / K * 1e3, "sampling_ms_per_step_rank0": t_sample / K * 1e3,
                "sampler_profile_us_per_env_step_rank0": sampler_profile},
        "gpu_launches": launches,
        "clocks": clk_value.summary(), "clocks_e2e": clk_e2e.summary(),
        "last_opt_info": {k: float(np.mean(getattr(info, k))) for k in info._fields},
    }
    if params_identical is not None:
        out["params_identical_across_ranks"] = params_identical

    # ---- roofline of the GAE scan kernel at the HBM-bound size, measured live (rank 0)
    if rank == 0:
        out["roofline"] = roofline_gae(U)
        try:   # the contraction kernels of the timed step; the largest one is the step's dominant kernel
            ks = step_kernel_rooflines()
            n_updates = int(PPO_KW.get("epochs", 4)) * int(PPO_KW.get("minibatches", 4))
            for k in ks:   # share of the timed step, to compare with the ncu launch list under profiles/
                k["share_of_step"] = k["us_per_launch"] * k["launches_per_update"] * n_updates / (out["ms_per_step"] * 1e3)
            out["step_kernels"] = ks
            out["roofline_step_kernel"] = max(ks, key=lambda k: k["share_of_step"])
        except Exception as e:  # never let the extra measurement break the bench line
            out["roofline_step_kernel"] = {"error": repr(e)[:200]}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"], out["gae_ppo_loss"] = cpu_baseline(U)
        gl = out["gae_ppo_loss"]
        gl["gpu_ms_inside_optimize_agent"] = in_situ_ms
        gl["speedup_inside_optimize_agent"] = gl["cpu_ms"] / in_situ_ms if in_situ_ms > 0 else None
        gl["note"] = ("gpu_ms_inside_optimize_agent: GAE + 16 fused-loss launches timed with CUDA events inside algo.optimize_agent "
                      "(the product path); gpu_ms_eager_wall_incl_python: the same kernels issued alone from Python, "
                      "where the ~25 us per call of ctypes + autograd bookkeeping is exposed")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        if args.dump_outputs:
            write_outputs(args.dump_outputs, dumps)
        print(json.dumps(out), flush=True)


DUMP_FRAMES = 16         # whole observation frames in the dump, drawn with a fixed seed from the [T,B] batch
DUMP_LIMIT = 64 << 20    # bytes


def _f(x):
    """Host copy as float32 / float64; integer and boolean arrays become float64 (exact)."""
    a = x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
    return a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)


def step_outputs(prefix, info, agent, samples=None):
    """What the last step of a timed loop handed its caller: ``optimize_agent``'s OptInfo rows and the parameters
    it updated, and for the end-to-end loop the batch ``obtain_samples`` returned.  The batch's observations
    (925 MB of frames) enter as every frame's byte sum plus DUMP_FRAMES whole frames."""
    out = {f"{prefix}_info_{k}": np.asarray(getattr(info, k), np.float64) for k in info._fields}
    out.update({f"{prefix}_param_{k}": _f(v) for k, v in agent.state_dict().items()})
    if samples is not None:
        a, e = samples.agent, samples.env
        obs = e.observation
        T, B = obs.shape[:2]
        pick = np.random.default_rng(0).choice(T * B, DUMP_FRAMES, replace=False)
        rows = torch.as_tensor(pick, device=obs.device)
        out.update({
            f"{prefix}_action": _f(a.action), f"{prefix}_prev_action": _f(a.prev_action),
            f"{prefix}_prob": _f(a.agent_info.dist_info.prob), f"{prefix}_value": _f(a.agent_info.value),
            f"{prefix}_bootstrap_value": _f(a.bootstrap_value), f"{prefix}_reward": _f(e.reward),
            f"{prefix}_prev_reward": _f(e.prev_reward), f"{prefix}_done": _f(e.done),
            f"{prefix}_observation_sum": _f(obs.sum(dim=tuple(range(2, obs.dim())), dtype=torch.float64)),
            f"{prefix}_observation_frames": obs.reshape(T * B, *obs.shape[2:])[rows].float().cpu().numpy(),
            f"{prefix}_observation_frame_index": pick.astype(np.float64)})
    return out


def write_outputs(path, arrays):
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT} byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def roofline_gae(U, T=128, B=1 << 20, reps=10):
    """Achieved HBM GB/s of the GAE streaming kernel: algorithmic bytes 17 B/element
    (r4 + v4 + done1 read, adv4 + ret4 written) + 4 B/column bootstrap, CUDA events on the launch
    stream, inputs (2.3 GB) far larger than L2."""
    peak, how = peaks()
    gen = torch.Generator(device="cuda").manual_seed(0)
    r = torch.randn(T, B, device="cuda", generator=gen)
    v = torch.randn(T, B, device="cuda", generator=gen)
    d = torch.rand(T, B, device="cuda", generator=gen) < 0.01
    b = torch.randn(1, B, device="cuda", generator=gen)
    adv, ret = torch.empty_like(r), torch.empty_like(r)
    fn = lambda: U.generalized_advantage_estimation(r, v, d, b, 0.99, 0.98, advantage_dest=adv, return_dest=ret, algo=1)
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    t = float(np.mean(ts))
    nbytes = T * B * 17 + 4 * B
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))["gae_stream_bytes_per_launch"]
    except Exception:
        pass
    return {"kernel": "returns_stream_kernel<4,GAE> [T=128, B=2^20]", "bound": "hbm", "achieved": nbytes / t / 1e9,
            "peak": peak, "unit": "GB/s", "frac": nbytes / t / 1e9 / peak, "traffic": traffic,
            "peak_source": how, "us_per_launch": t * 1e6, "algorithmic_bytes": nbytes}


def step_kernel_rooflines(N=8192, reps=10):
    """The contraction kernels of one minibatch update (N = 8192 samples, (4,84,84) frames), each timed alone with
    CUDA events on the launch stream, with its algorithmic bytes (what has to cross HBM once) against the HBM
    roof - and, for the fully connected layer, its useful flops against the TF32 tensor roof.  The caller picks
    the largest one as ``roofline_step_kernel``."""
    from rlpyt_b200 import _lib
    from rlpyt_b200.models.conv2_op import wgrad_scratch
    from rlpyt_b200.models.gemm_op import gemm_tn
    peak, how = peaks()
    lib = _lib.load()
    gen = torch.Generator(device="cuda").manual_seed(1)
    obs = torch.randint(0, 256, (4 * N,) + IMAGE, dtype=torch.uint8, device="cuda", generator=gen)   # 925 MB > L2
    rows = torch.randperm(4 * N, device="cuda", generator=gen)[:N].contiguous()
    oh, ow = (IMAGE[1] - 8) // 4 + 1, (IMAGE[2] - 8) // 4 + 1
    o1 = torch.randn(N, 16, oh, ow, device="cuda", generator=gen)
    g1 = torch.randn(N, 16, oh, ow, device="cuda", generator=gen)
    x2 = torch.relu(o1)
    oh2, ow2 = (oh - 2) // 2 + 1, (ow - 2) // 2 + 1
    o2 = torch.randn(N, 32, oh2, ow2, device="cuda", generator=gen)
    g2 = (torch.randn(N, 32, oh2, ow2, device="cuda", generator=gen) * (o2 > 0)).contiguous()
    w1, b1 = torch.randn(16, 4, 8, 8, device="cuda", generator=gen) / 16, torch.randn(16, device="cuda", generator=gen)
    w2, b2 = torch.randn(32, 16, 4, 4, device="cuda", generator=gen) / 16, torch.randn(32, device="cuda", generator=gen)
    gw1, gb1 = torch.empty_like(w1), torch.empty_like(b1)
    gw2, gb2 = torch.empty_like(w2), torch.empty_like(b2)
    gx2 = torch.empty_like(x2)
    y1, y2 = torch.empty_like(o1), torch.empty_like(o2)
    sc_i8 = torch.empty(int(lib.rl_conv1_u8_wgrad_i8_scratch_bytes()) // 4 + 4, device="cuda")
    sc_tc = wgrad_scratch(obs.device)
    sc_dg = torch.empty(int(lib.rl_conv2_dgrad_tc_scratch_bytes()) // 4 + 4, device="cuda")
    sc_w2 = torch.empty(int(lib.rl_conv2_wgrad_s2d_scratch_bytes()) // 4 + 4, device="cuda")
    fa = torch.randn(N, 3200, device="cuda", generator=gen)
    fb = torch.randn(512, 3200, device="cuda", generator=gen)
    amax1 = g1.abs().amax(dim=(0, 2, 3)).contiguous()        # what rl_conv2_dgrad_s2d_absmax hands to the first layer's weight gradient
    amax2 = torch.empty(16, device="cuda")
    C, H, W = IMAGE
    P1, P2 = 16 * oh * ow * 4, 32 * oh2 * ow2 * 4
    i8 = bool(lib.rl_conv1_u8_i8_supported(C, H, W))
    s2d = bool(lib.rl_conv2_s2d_supported(16, oh, ow))
    kernels = [
        (("conv1_i8_wgrad_kernel + reduce (kind::i8; channel maxima handed over by conv2's input-gradient epilogue)" if i8
          else "conv_wgrad_tc_kernel<Layer1>") + " [N=8192, (4,84,84) u8]",
         (lambda: _lib.call("rl_conv1_u8_wgrad_i8_scaled", _lib.ptr(obs), _lib.ptr(rows), _lib.ptr(o1), _lib.ptr(g1), _lib.ptr(amax1),
                            _lib.ptr(gw1), _lib.ptr(gb1), N, C, H, W, _lib.ptr(sc_i8), _lib.stream(), n_launch=2)) if i8 else
         (lambda: _lib.call("rl_conv1_u8_wgrad_tc", _lib.ptr(obs), _lib.ptr(rows), _lib.ptr(o1), _lib.ptr(g1), _lib.ptr(gw1),
                            _lib.ptr(gb1), N, C, H, W, _lib.ptr(sc_tc), _lib.stream(), n_launch=2)),
         N * (C * H * W + 2 * P1), "conv1_wgrad_bytes_per_launch"),
        (("conv1_i8_fwd_kernel (kind::i8)" if i8 else "conv_fwd_tc_kernel<Layer1>") + " [N=8192]",
         lambda: _lib.call("rl_conv1_u8_forward_i8" if i8 else "rl_conv1_u8_forward_tc", _lib.ptr(obs), _lib.ptr(rows), _lib.ptr(w1),
                           _lib.ptr(b1), _lib.ptr(y1), N, C, H, W, 1, _lib.stream()),
         N * (C * H * W + P1), "conv1_fwd_bytes_per_launch"),
        (("conv2_s2d_fwd_kernel" if s2d else "conv_fwd_tc_kernel<Layer2>") + " [N=8192]",
         lambda: _lib.call("rl_conv2_forward_s2d" if s2d else "rl_conv2_forward_tc", _lib.ptr(x2), _lib.ptr(w2), _lib.ptr(b2), _lib.ptr(y2),
                           N, 16, oh, ow, 1, _lib.stream()),
         N * (P1 + P2), "conv2_fwd_bytes_per_launch"),
        (("conv2_s2d_dgrad_kernel (+ per-channel |gradient| maxima)" if s2d else "conv_fwd_tc_kernel<Dgrad2>") + " [N=8192]",
         (lambda: _lib.call("rl_conv2_dgrad_s2d_absmax", _lib.ptr(g2), _lib.ptr(w2), _lib.ptr(gx2), _lib.ptr(amax2), N, 16, oh, ow,
                            _lib.stream())) if s2d else
         (lambda: _lib.call("rl_conv2_dgrad_tc", _lib.ptr(g2), _lib.ptr(w2), _lib.ptr(gx2), N, 16, oh, ow, _lib.ptr(sc_dg), _lib.stream(),
                            n_launch=2)),
         N * (P1 + P2), "conv2_dgrad_bytes_per_launch"),
        (("conv2_s2d_wgrad_kernel + reduce" if s2d else "conv_wgrad_tc_kernel<Layer2>") + " [N=8192]",
         (lambda: _lib.call("rl_conv2_wgrad_s2d", _lib.ptr(x2), _lib.ptr(g2), _lib.ptr(gw2), _lib.ptr(gb2), N, 16, oh, ow, _lib.ptr(sc_w2),
                            _lib.stream(), n_launch=2)) if s2d else
         (lambda: _lib.call("rl_conv2_wgrad_tc", _lib.ptr(x2), None, _lib.ptr(g2), _lib.ptr(gw2), _lib.ptr(gb2), N, 16, oh, ow,
                            _lib.ptr(sc_tc), _lib.stream(), n_launch=2)),
         N * (P1 + P2), "conv2_wgrad_bytes_per_launch"),
    ]
    try:
        traffic_tab = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
    except Exception:
        traffic_tab = {}
    out = []
    for name, fn, nbytes, tkey in kernels:
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e-3)
        t = float(np.mean(ts))
        out.append({"kernel": name, "bound": "hbm", "achieved": nbytes / t / 1e9, "peak": peak, "unit": "GB/s",
                    "frac": nbytes / t / 1e9 / peak, "traffic": traffic_tab.get(tkey), "peak_source": how,
                    "us_per_launch": t * 1e6, "algorithmic_bytes": nbytes, "launches_per_update": 1})
    # fully connected layer: 3 GEMMs per update (forward, input gradient, weight gradient), 2*8192*512*3200 flops each,
    # on the kernel the Linear op dispatches (csrc/gemm_ts.cuh, incl. the preparation of its small operand)
    from rlpyt_b200.models import gemm_op
    ts_impl = gemm_op._use_ts(N)
    fg = torch.randn(N, 512, device="cuda")

    def fc_fwd():
        return gemm_op.gemm_ts(fa, fb, gemm_op.split_lo(fb), None, True) if ts_impl else gemm_tn(fa, fb)

    def fc_dgrad():
        return gemm_op.gemm_ts(fg, *gemm_op.transpose_split(fb)) if ts_impl else gemm_tn(fg, gemm_op.transpose2d(fb))

    def fc_wgrad():
        if ts_impl:
            return gemm_op.gemm_ts(fa, *gemm_op.transpose_split(fg), a_mmajor=True, c_trans=True)
        return gemm_tn(gemm_op.transpose2d(fg), gemm_op.transpose2d(fa))

    try:
        tf32_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"]) / 2
        tsrc = "measured bf16 cuBLAS TF/s / 2 (TF32 runs at half the bf16 rate)"
    except Exception:
        tf32_peak, tsrc = 1125.0, "nominal dense TF32 (B200_PROFILING.md)"
    fl = 2.0 * N * 512 * 3200
    kname = "gemm_ts_kernel" if ts_impl else "gemm_tf32x3_kernel"
    for what, fn in (("forward 8192x512x3200", fc_fwd), ("input gradient 8192x3200x512", fc_dgrad),
                     ("weight gradient 3200x512x8192", fc_wgrad)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e-3)
        t = float(np.mean(ts))
        out.append({"kernel": "%s [fc %s, fp32-accurate 3xTF32, incl. operand preparation]" % (kname, what), "bound": "tensor",
                    "achieved": fl / t / 1e12, "peak": tf32_peak, "unit": "TFLOP/s", "frac": fl / t / 1e12 / tf32_peak,
                    "issued_frac": 3 * fl / t / 1e12 / tf32_peak,
                    "traffic": traffic_tab.get("gemm_fc_bytes_per_launch"), "peak_source": tsrc, "us_per_launch": t * 1e6,
                    "algorithmic_flops": fl, "issued_flops": 3 * fl, "launches_per_update": 1,
                    "note": "achieved/frac count useful fp32-equivalent flops; the 3-term split issues 3x as many on the "
                            "tensor pipe (issued_frac)"})
    return out


def cpu_baseline(U):
    """Rank 0, N=1: (i) the reference arm (``--impl reference``: the unmodified reference from oracle/_ref on
    this box's host cores, bounded sample, same config) run as a child process for a few steps - its line's
    ``value`` (learner only) and ``e2e`` (sampler + learner) are what ``value`` / ``e2e`` above compare with;
    (ii) the north_star unit "reference CPU GAE + PPO-loss" at [128,256] (GAE on torch-CPU tensors + 16 x loss
    fwd+bwd arithmetic at N=8192) next to the same work on the GPU kernels."""
    from oracle import pg_loss  # noqa: F401  (checker side only; see oracle/__init__.py)
    from oracle.ppo import gae_plus_loss_cpu
    from rlpyt_b200.algos.pg import loss_ops
    threads = torch.get_num_threads()
    rng = np.random.default_rng(0)
    base = {"value": None, "unit": "env-steps/s", "cores": threads, "kind": "reference", "sample": "unavailable"}
    try:
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3", "--warmup", "1",
                            "--no-gpu-context"], capture_output=True, text=True, timeout=600,
                           env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
        line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1]
        ref = json.loads(line)
        base = dict(ref["cpu_baseline"])
        base["e2e_value"] = ref["e2e"]["value"]
        base["learner_only_value"] = ref["value"]
    except Exception as e:  # noqa: BLE001 - the baseline must never break the bench line
        base["error"] = repr(e)[:300]

    # (ii) GAE + 16 x PPO-loss, CPU reference arithmetic vs the GPU kernels, full [128,256] size
    T, B, N, A = T_CFG, B_CFG, 8192, N_ACTIONS
    r = rng.standard_normal((T, B)).astype(np.float32)
    v = rng.standard_normal((T, B)).astype(np.float32)
    d = rng.random((T, B)) < 0.01
    b = rng.standard_normal((1, B)).astype(np.float32)
    p_new = rng.dirichlet(np.ones(A), N).astype(np.float32)
    p_old = rng.dirichlet(np.ones(A), N).astype(np.float32)
    case = (p_new, rng.standard_normal(N).astype(np.float32), p_old, rng.integers(0, A, N),
            rng.standard_normal(N).astype(np.float32), rng.standard_normal(N).astype(np.float32), None, 0.1, 1.0, 0.01)
    gae_plus_loss_cpu(r, v, d, b, 0.99, 0.98, case)
    reps = 10
    t0 = time.perf_counter()
    for _ in range(reps):
        gae_plus_loss_cpu(r, v, d, b, 0.99, 0.98, case)
    cpu_ms = (time.perf_counter() - t0) / reps * 1e3
    cu = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    rc, vc, dc, bc = cu(r), cu(v), cu(d), cu(b)
    adv, ret = torch.empty_like(rc), torch.empty_like(rc)
    pn, vv, po, ac, Rc, Ac = (cu(x) for x in case[:6])

    def gpu_unit():
        U.generalized_advantage_estimation(rc, vc, dc, bc, 0.99, 0.98, advantage_dest=adv, return_dest=ret)
        for _ in range(16):
            p = pn.detach().requires_grad_(True)
            q = vv.detach().requires_grad_(True)
            loss, _sc = loss_ops.ppo_loss(p, q, po, ac, Rc, Ac, None, 0.1, 1.0, 0.01)
            loss.backward()
    for _ in range(3):
        gpu_unit()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(20):
        gpu_unit()
    torch.cuda.synchronize()
    gpu_ms = (time.perf_counter() - t0) / 20 * 1e3
    # the same 1 + 16 x 4 launches captured once and replayed as a CUDA graph (how a deployment would
    # issue a fixed-shape unit): wall time == device time, no per-call Python / ctypes cost
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gpu_unit()
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    graph_ms = e0.elapsed_time(e1) / 50
    unit = {"what": "GAE [128,256] + 16 x PPO-loss fwd+bwd (N=8192, A=6), no network", "cpu_ms": cpu_ms,
            "gpu_ms_cuda_graph": graph_ms, "speedup": cpu_ms / graph_ms,
            "gpu_ms_eager_wall_incl_python": gpu_ms, "speedup_eager": cpu_ms / gpu_ms, "cpu_threads": threads}
    return base, unit


# --------------------------------------------------------------------------------------------- reference arm
REF_T = 16     # bounded sample of the reference arm: [T=16, B=256] per step (B, minibatch structure, env, workers as configured)


def _reference_affinity(world):
    from rlpyt_b200.utils.affinity import make_affinity
    try:
        aff = make_affinity(0, None, local_rank=0, ranks_per_node=1, node_share=8)
        return [c[0] for c in aff["workers_cpus"]]
    except Exception:  # noqa: BLE001
        return list(range(max(1, (os.cpu_count() or 2) // 8 - 1)))


def run_reference(args):
    """``--impl reference``: the UNMODIFIED reference (oracle/_ref, copied there by oracle/reference_install.py)
    through its own API - ``GpuSampler`` with ``cuda_idx=None`` (batched action serving on torch-CPU
    with every host thread, env stepping in forked workers pinned to the same cores this repo's arm uses) +
    ``PPO.optimize_agent`` on torch-CPU - baseline/reference_arm.py.  Same config as the b200 arm (B=256, the
    same PPO hyper-parameters, env and worker cores); each step is a bounded sample [T=16, B=256] of the
    [T=128, B=256] iteration (4096 of 32768 env-steps: per-env-step cost does not depend on T).
    ``value`` = learner only (optimize_agent), ``e2e`` = sampler + learner: like for like with the b200 line.
    Falls back to the oracle port when oracle/_ref is absent."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K, W = args.steps, args.warmup
    threads = torch.get_num_threads()
    from baseline import reference_arm as R
    if not R.available():
        return run_reference_port(args)
    workers_cpus = _reference_affinity(1)
    real_stdout = sys.stdout
    sys.stdout = sys.stderr          # the reference's logger prints to stdout; this arm's stdout is ONE JSON line
    loop = R.ReferenceLoop(REF_T, B_CFG, ENV_KW, PPO_KW, workers_cpus=workers_cpus, cuda_idx=None, seed=0)
    try:
        for _ in range(W):
            loop.step()
        loop.reset_timers()
        t0 = time.perf_counter()
        for _ in range(K):
            loop.step()
        dt = time.perf_counter() - t0
        t_opt, t_smp = loop.t_optimize, loop.t_sample
    finally:
        loop.shutdown()
    steps = REF_T * B_CFG
    val_e2e, val_learn = steps * K / dt, steps * K / t_opt
    sample = (f"unmodified reference (oracle/_ref): GpuSampler(cuda_idx=None, {len(workers_cpus)} worker processes) + "
              f"PPO on torch-CPU fp32, {threads} threads; bounded sample [T={REF_T},B={B_CFG}] per step "
              f"({steps} of {T_CFG * B_CFG} env-steps), minibatches=4 epochs=4")
    out = {
        "impl": "reference", "metric": "env-steps/sec PPO Atari [T=128,B=256] at 1/2/4/8 GPU; GAE-scan GB/s",
        "value": val_learn, "unit": "env-steps/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": K, "warmup": W,
        "ms_per_step": t_opt / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "value_scope": "learner only: PPO.optimize_agent on torch-CPU (compare with the b200 line's value)",
        "config": {"workload": "PPO+AtariFfAgent, synthetic Atari env obs (4,84,84) u8, B=256 per GPU, gamma .99 lambda .98 "
                               "lr 1e-3 clip .1 4x4 (the b200 arm's config)", "sample": sample,
                   "env_workers": len(workers_cpus)},
        "cpu_baseline": {"value": val_e2e, "unit": "env-steps/s", "cores": threads, "kind": "reference", "sample": sample},
        "e2e": {"value": val_e2e, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "ms_per_step": dt / K * 1e3, "sampling_ms_per_step": t_smp / K * 1e3},
        "gpu_launches": 0,
    }
    # context (SURVEY 8(d) row 3): the same reference objects with cuda_idx=0 = stock PyTorch/cuDNN/cuBLAS on the B200,
    # full [T=128, B=256] iterations
    if not args.no_gpu_context and out["n_gpus"] == 1 and torch.cuda.is_available():
        try:
            g = R.ReferenceLoop(T_CFG, B_CFG, ENV_KW, PPO_KW, workers_cpus=workers_cpus, cuda_idx=0, seed=0)
            try:
                for _ in range(2):
                    g.step()
                g.reset_timers()
                t0 = time.perf_counter()
                n = 4
                for _ in range(n):
                    g.step()
                gdt = time.perf_counter() - t0
                out["stock_pytorch_gpu"] = {
                    "what": "unmodified reference with cuda_idx=0 (stock PyTorch kernels on this B200), [T=128,B=256], "
                            f"{n} iterations", "e2e_value": T_CFG * B_CFG * n / gdt, "unit": "env-steps/s",
                    "learner_only_value": T_CFG * B_CFG * n / g.t_optimize, "ms_per_step": gdt / n * 1e3,
                    "sampling_ms_per_step": g.t_sample / n * 1e3, "optimize_ms_per_step": g.t_optimize / n * 1e3}
            finally:
                g.shutdown()
        except Exception as e:  # noqa: BLE001
            out["stock_pytorch_gpu"] = {"error": repr(e)[:300]}
    sys.stdout = real_stdout
    print(json.dumps(out), flush=True)


def run_reference_port(args):
    """Fallback when oracle/_ref is missing: the oracle port (serial CPU rollout + PPO on torch-CPU)."""
    from oracle import atari_ff
    from oracle.collector import SerialRollout
    from oracle.ppo import PpoOracle
    from rlpyt_b200.envs.synthetic import SyntheticAtariEnv
    threads = torch.get_num_threads()
    Tb, Bb = REF_T, B_CFG
    np.random.seed(0)
    torch.manual_seed(0)
    envs = [SyntheticAtariEnv(**ENV_KW) for _ in range(Bb)]
    for i, e in enumerate(envs):
        e.seed(1 + i)
    sd = atari_ff.init_state_dict(IMAGE, N_ACTIONS, 0)
    algo = PpoOracle(sd, n_itr=10 ** 6, **PPO_KW)
    roll = SerialRollout(envs, sd, Tb, N_ACTIONS)
    t_opt = [0.0]

    def step(itr):
        buf = roll.collect_batch(algo.state_dict())
        t0 = time.perf_counter()
        r = algo.optimize_agent(itr, buf["observation"], buf["all_action"][1:], buf["all_reward"][1:], buf["done"],
                                buf["value"], buf["prob"], buf["bootstrap_value"])
        t_opt[0] += time.perf_counter() - t0
        return r
    K, W = args.steps, args.warmup
    for i in range(W):
        step(i)
    t_opt[0] = 0.0
    t0 = time.perf_counter()
    for i in range(K):
        step(W + i)
    dt = time.perf_counter() - t0
    val = Tb * Bb * K / dt
    sample = (f"oracle port (serial collector + PPO, torch-CPU fp32, {threads} threads; oracle/_ref missing), bounded sample "
              f"[T={Tb},B={Bb}] per step ({Tb * Bb} of {T_CFG * B_CFG} env-steps)")
    print(json.dumps({
        "impl": "reference", "metric": "env-steps/sec PPO Atari [T=128,B=256] at 1/2/4/8 GPU; GAE-scan GB/s",
        "value": Tb * Bb * K / t_opt[0], "unit": "env-steps/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": K,
        "warmup": W, "ms_per_step": t_opt[0] / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "value_scope": "learner only (oracle port)",
        "config": {"workload": "PPO+AtariFf on CPU (reference algorithm), synthetic Atari env obs (4,84,84) u8", "sample": sample},
        "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workers", type=int, default=0, help="env workers per rank (0 = one per physical core of the share)")
    ap.add_argument("--workers-per-core", type=int, default=2, help="env workers per physical core of the rank's share (1 or 2)")
    ap.add_argument("--sampler", default="alternating", choices=["alternating", "gpu"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-context", action="store_true", help="reference arm: skip the stock-PyTorch-on-GPU context leg")
    ap.add_argument("--workload", default="ppo", choices=["ppo", "gae", "replay", "dqn"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last step of each timed loop computed to DIR/<name>.npy (ppo workload, b200 arm)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.workload != "ppo" or args.impl != "b200"):
        ap.error("--dump-outputs is implemented for the ppo workload of the b200 arm")
    if args.workload != "ppo":
        from tools import workload_benches
        return workload_benches.run(args)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
