#!/usr/bin/env python
"""Headline benchmark: env steps/sec of the PPO hot path (BASELINE.json metric) on N B200s.

    python bench.py --gpus 1 --steps K --warmup W            # our arm (libb200rl kernels)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: the reference's CPU path
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...   (N > 1; one rank per GPU, NCCL)

Workload (config.workload): ppo_atari_envpool at BASELINE.json configs[1] -- per GPU num_envs=1024,
num_steps=128 (131 072 env steps per iteration), 4 epochs x 4 minibatches of 32 768, NatureCNN,
Breakout-shaped SYNTHETIC vector env (no envpool/ALE in the image).  A "step" of this benchmark is
one PPO iteration = rollout (128 policy steps) + bootstrap + GAE + 16 minibatch updates.

  value : whole-job SPS with the observation batches already resident in HBM (no host round trips)
  e2e   : the same metric through the public loop (PPOEngine as the drop-in scripts drive it) with
          HOST buffers: every policy step copies the pinned uint8 batch H2D and the actions D2H,
          rewards/dones go up once per iteration, losses come back once per iteration.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path
from types import SimpleNamespace

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "env steps/sec (SPS) PPO Breakout num_envs=1024"
FLOP_PER_ENV_STEP = 243.1e6     # SURVEY.md 8(d): fwd 18.69 MFLOP x [129/128 + 4 epochs x 3]
HBM_BYTES_PER_ENV_STEP = 169344  # uint8 frame x [1 H2D write + 1 rollout read + 4 epoch reads]


def bench_config(N, T, world):
    """`config` of the JSON line: identical for our arm and for the reference arm (same workload, same shapes)."""
    return {"workload": "ppo_atari_envpool Breakout-shaped synthetic vec env; per GPU num_envs=%d num_steps=%d, "
                        "4 epochs x 4 minibatches of %d, NatureCNN A=4; one step = one PPO iteration" % (N, T, N * T // 4),
            "global_num_envs": N * world, "parallelism": f"dp{world}",
            "timing": "inputs_larger_than_L2 (3.7 GB uint8 rollout + 2.8 GB activations per minibatch vs 126 MB L2)",
            "gae_kernel": "scan"}


def ppo_args(num_envs, num_steps, num_iterations, precision):
    """Reference defaults of ppo_atari_envpool.py:19-80."""
    a = SimpleNamespace(
        seed=1, learning_rate=2.5e-4, num_envs=num_envs, num_steps=num_steps, anneal_lr=True, gamma=0.99,
        gae_lambda=0.95, num_minibatches=4, update_epochs=4, norm_adv=True, clip_coef=0.1, clip_vloss=True,
        ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5, target_kl=None, precision=precision)
    a.batch_size = num_envs * num_steps
    a.minibatch_size = a.batch_size // a.num_minibatches
    a.num_iterations = num_iterations
    return a


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []                # (arrival time, csv line)
        self.t0 = self.t1 = None

    def start(self):
        """Start sampling (nvidia-smi needs ~0.5 s to deliver its first line: start it BEFORE the warm-up).  200 ms is the
        recipe's period (B200_PROFILING.md); every query takes driver locks, and at 50 ms the end-to-end rollout -- which is
        bound by host-side CUDA API calls -- measurably slowed down."""
        period = os.environ.get("BENCH_CLOCK_SAMPLE_MS", "200")
        if period == "0":
            self.proc = None
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", period],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.21)               # let the sample that covers the end of the region arrive
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smmax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = [ln for ts, ln in self.lines if self.t0 is None or (self.t0 <= ts <= (self.t1 or ts) + 0.2)]
        window = "timed region"
        if not lines and self.lines:   # region shorter than one sampling period: the sample nearest to it
            mid = 0.5 * (self.t0 + (self.t1 or self.t0))
            lines = [min(self.lines, key=lambda x: abs(x[0] - mid))[1]]
            window = "nearest sample"
        for ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smmax.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smmax) if smmax else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


def pin_to_gpu_cores(gpu_index):
    """Run this process (and the threads it creates later: the engine's host worker pools) on the CPU cores NVML reports as
    local to the GPU, so that pinned staging memory, the env buffers and the upload path sit on the GPU's NUMA node.  One
    process per GPU: every rank pins to its own GPU's cores.  OFF by default (BENCH_CPU_AFFINITY=1 turns it on): on the
    shared hosts this was measured on, the GPU-local socket is where every other tenant's processes sit as well, and the
    pinned run was 2x slower than letting the scheduler pick idle cores (profiles/r2_host_sensitivity.md)."""
    if os.environ.get("BENCH_CPU_AFFINITY", "0") != "1" or not hasattr(os, "sched_setaffinity"):
        return None
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if len(cpus) >= 4:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        return None
    return None


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, eng, stats):
    """Write what the last timed iteration of `value` hands its caller as float32 DIR/<name>.npy: the rollout's actions,
    log-probabilities and values, the GAE advantages and returns, the bootstrap values, the loss statistics of every
    minibatch update and the updated flat parameter vector.  Inputs are seeded, so two builds run with the same arguments
    can be compared file by file.  Above DUMP_BYTES in all, the [num_steps, num_envs] arrays keep a fixed, seeded subset
    of env columns."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    rollout = {"actions": eng.actions, "logprobs": eng.logprobs, "values": eng.values, "advantages": eng.advantages,
               "returns": eng.returns}
    flat = {"next_value": eng.next_value, "params": eng.flat.flat}
    T, N = eng.T, eng.N
    headers = 4096                                 # .npy headers, 128 bytes per file
    room = (DUMP_BYTES - headers - 4 * sum(t.numel() for t in flat.values()) - stats["per_update"].nbytes) // (4 * len(rollout) * T)
    cols = slice(None) if room >= N else np.sort(np.random.default_rng(0).choice(N, max(int(room), 1), replace=False))
    for name, t in rollout.items():
        np.save(out / f"{name}.npy", t.float().cpu().numpy()[:, cols])
    for name, t in flat.items():
        np.save(out / f"{name}.npy", t.float().cpu().numpy())
    np.save(out / "update_stats.npy", stats["per_update"].astype(np.float32))


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        z = json.loads(p.read_text())
        return z.get("bf16_tflops_sustained", 1400.0), z.get("hbm_gbs", 6650.0), "measured"
    return 1400.0, 6650.0, "fallback"


# --------------------------------------------------------------------------------- our arm
def run_ours(opt):
    import torch
    import torch.distributed as dist
    from cleanrl_b200 import _lib, build, ops
    from cleanrl_b200.agents import NatureCNNAgent
    from cleanrl_b200.ppo_engine import PPOEngine
    from cleanrl_b200.synthetic_envs import SyntheticAtariVec

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl=ours) needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    pinned_cores = pin_to_gpu_cores(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    build.build()
    lib = _lib.load()

    N, T, K, W = opt.num_envs, opt.num_steps, opt.steps, opt.warmup
    total_iters = 5 * (K + W) + 8                # up to five timed loops (resident, profiled, whole-upload, e2e): lr stays > 0
    args = ppo_args(N, T, total_iters, opt.precision)
    seed = args.seed + rank                      # per-rank env / numpy streams (ppo_atari_multigpu.py:208-210)
    np.random.seed(seed)
    torch.manual_seed(args.seed)                  # identical initial weights on every rank (:211)
    envs = SyntheticAtariVec(N, seed=seed, mode="pool", pinned=True)
    envs.single_observation_space, envs.single_action_space = envs.observation_space, envs.action_space
    agent = NatureCNNAgent(envs).to(device)
    agent.precision = opt.precision
    torch.manual_seed(seed)
    all_reduce = (lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM)) if world > 1 else None
    eng = PPOEngine(agent, args, envs.observation_space.shape, np.uint8, N, device, world_size=world,
                    gae_mode=1, all_reduce=all_reduce)

    def replica_trace(tag):
        """BENCH_REPLICA_TRACE=1: after which phase do the replicas stop being bit-identical (diagnostic, stderr)."""
        if not os.environ.get("BENCH_REPLICA_TRACE"):
            return
        torch.cuda.synchronize()
        res_ = []
        L = eng.agent._tc_plan()
        for nm, buf in (("params", eng.flat.flat), ("grad", eng.flat.grad), ("exp_avg", eng.flat.exp_avg), ("exp_avg_sq", eng.flat.exp_avg_sq)):
            bad = ~torch.isfinite(buf)
            nbad = int(bad.sum())
            first = [int(i) for i in bad.nonzero().flatten()[:6]] if nbad else []
            same = None
            if world > 1:
                ref = buf.clone()
                dist.broadcast(ref, 0)
                same = bool(torch.equal(torch.nan_to_num(ref, nan=12345.0), torch.nan_to_num(buf, nan=12345.0)))
            res_.append((nm, "nonfinite", nbad, first, "same_as_rank0", same))
        print(f"[replica_trace rank {rank}] {tag}: step={eng.flat.step} numel={eng.flat.flat.numel()} {res_}", file=sys.stderr, flush=True)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    it_counter = [0]

    def lr_now():
        it_counter[0] += 1
        return (1.0 - (it_counter[0] - 1.0) / total_iters) * args.learning_rate

    # ---- e2e: the public loop with host buffers.  --env-groups G > 1 (default 2): PPOEngine.collect over G independent
    #      vector envs, software-pipelined (what `ppo_atari_envpool.py --env-groups G` runs); 1: the reference's loop order
    #      Observations: `--env-obs stack` (default) = frame-stacked like envpool's stack_num=4 Atari observation (planes 0..2 of
    #      an env's observation are planes 1..3 of its previous one; done envs come back with 4 fresh planes), so the engine's
    #      frame-stack delta upload applies; `pool` = unrelated random batches every step (every observation goes up whole).
    G = max(1, int(opt.env_groups))
    env_sets = {}

    def use_envs(mode):
        if mode not in env_sets:
            parts = [SyntheticAtariVec(N // G, seed=seed + g * (N // G), mode=mode, pinned=True) for g in range(G)]
            env_sets[mode] = (parts, {"obs": [e.reset() for e in parts], "done": [np.zeros(N // G, dtype=np.float32) for _ in parts]})
        return env_sets[mode]

    # frame-stacked observations only pay off through the delta upload; where the engine uploads whole observations (several
    # ranks per host by default, CLEANRL_B200_DELTA_UPLOAD=0) the e2e arm hands it dense pinned batches as rounds 1-2 did
    obs_mode = opt.env_obs if (opt.env_obs == "pool" or eng.delta_upload) else "pool"
    if G > 1:
        env_parts, state = use_envs(obs_mode)
    else:
        state = {"obs": envs.reset(), "done": np.zeros(N, dtype=np.float32)}

    phase_ev = []                                  # (start, rollout done, update done) events per e2e iteration

    def iteration_e2e():
        if G > 1:
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            evs[0].record()
            obs_p, done_p = eng.collect(env_parts, state["obs"], state["done"])
            eng.finish_rollout_parts(obs_p, done_p)
            evs[1].record()
            st = eng.update(lr_now())
            evs[2].record()
            phase_ev.append(evs)
            state["obs"], state["done"] = obs_p, done_p
            return st
        next_obs, next_done = state["obs"], state["done"]
        for step in range(T):
            action = eng.policy_step(step, next_obs, next_done)
            next_obs, reward, next_done, info = envs.step(action)
            eng.record_reward(step, reward)
        eng.finish_rollout(next_obs, next_done)
        st = eng.update(lr_now())
        state["obs"], state["done"] = next_obs, next_done
        return st

    # ---- resident: observation batches, rewards and dones already in HBM
    pool_dev = torch.from_numpy(envs._batches).to(device)
    g = torch.Generator(device="cpu").manual_seed(seed)
    eng_rewards = torch.randint(0, 2, (T, N), generator=g).float().to(device)
    eng_dones = (torch.rand(T, N, generator=g) < 0.02).float().to(device)

    def iteration_resident():
        P = pool_dev.shape[0]
        if eng.cuda_graphs and getattr(agent, "graph_friendly", False):
            eng.rollout_resident(pool_dev)          # all T steps = one graph launch (no host launch per step)
        else:
            for step in range(T):
                eng.policy_step_resident(step, pool_dev[step % P])
        eng.rewards.copy_(eng_rewards)
        eng.dones.copy_(eng_dones)
        if eng.s2d:
            eng._to_storage(pool_dev[T % P], None)
        else:
            eng.next_obs.copy_(pool_dev[T % P])
        eng.finish_rollout(None, None, resident=True)
        return eng.update(lr_now())

    def timed(fn, profile=False):
        sampler = ClockSampler(local_rank)
        sampler.start()
        for _ in range(W):
            fn()
        barrier()
        sampler.mark_begin()
        h2d0, d2h0, l0 = eng.h2d_bytes, eng.d2h_bytes, lib.b200rl_launch_count() + eng.graph_launches
        if profile:
            lib.b200rl_profile_reset()
            lib.b200rl_profile_enable(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        st = None
        for _ in range(K):
            st = fn()
        e1.record()
        torch.cuda.synchronize()
        sampler.mark_end()
        ms = e0.elapsed_time(e1)
        prof = None
        if profile:
            lib.b200rl_profile_enable(0)
            import ctypes
            cbuf = ctypes.create_string_buffer(1 << 16)
            _lib.check(lib.b200rl_profile_summary(cbuf, 1 << 16), "profile_summary")
            prof = json.loads(cbuf.value.decode())
        barrier()
        clocks = sampler.stop()
        t = torch.tensor([ms], device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return dict(ms=float(t.item()), h2d=(eng.h2d_bytes - h2d0) / K, d2h=(eng.d2h_bytes - d2h0) / K,
                    launches=lib.b200rl_launch_count() + eng.graph_launches - l0, clocks=clocks, stats=st, prof=prof)

    def phases(r):
        if phase_ev:                               # where an end-to-end iteration goes (device time, the K timed iterations)
            torch.cuda.synchronize()
            last = phase_ev[-K:]
            r["rollout_ms"] = sum(a.elapsed_time(b) for a, b, _ in last) / K
            r["update_ms"] = sum(b.elapsed_time(c) for _, b, c in last) / K
        return r

    replica_trace("init")
    res = timed(iteration_resident)                 # `value`: update replayed as per-epoch CUDA graphs, no profiling events
    if opt.dump_outputs and rank == 0:
        dump_outputs(opt.dump_outputs, eng, res["stats"])
    replica_trace("after resident loop")
    eng.update_graphs = False                       # per-kernel CUDA-event brackets cannot live inside a captured graph:
    prof_run = timed(iteration_resident, profile=True)      # the kernel table comes from an eager pass of the same iteration
    eng.update_graphs = os.environ.get("CLEANRL_B200_UPDATE_GRAPHS", "1") != "0"
    replica_trace("after profiled resident loop")
    res["prof"] = prof_run["prof"]
    res["eager_ms"] = prof_run["ms"]
    e2e_whole = None
    if G > 1 and obs_mode == "stack" and eng.delta_upload and not opt.no_whole_upload_arm:
        # secondary arm: the same loop on unrelated observations, every one uploaded whole (round 2's headline path)
        env_parts, state = use_envs("pool")
        eng.delta_upload = False
        e2e_whole = phases(timed(iteration_e2e))
        replica_trace("after whole-upload e2e loop")
        eng.delta_upload = True
        env_parts, state = use_envs("stack")
    ff0, rd0 = eng.delta_full_frames, eng.delta_redos
    host_acc = None
    if os.environ.get("BENCH_E2E_BREAKDOWN") and G > 1:      # diagnostic: host wall time per group step (adds ~1 us per call)
        host_acc = {"wait": 0.0, "env": 0.0, "launch": 0.0}

        def _wrap(obj, name, key):
            f = getattr(obj, name)

            def g(*a, **k):
                t0 = time.perf_counter()
                r = f(*a, **k)
                host_acc[key] += time.perf_counter() - t0
                return r
            setattr(obj, name, g)
        _wrap(eng, "wait_actions", "wait"); _wrap(eng, "launch_part", "launch")
        for e in env_parts:
            _wrap(e, "step", "env")
    e2e = phases(timed(iteration_e2e))
    if host_acc is not None:
        e2e["host_us_per_env_step"] = {k: round(v / ((W + K) * T) * 1e6, 1) for k, v in host_acc.items()}
    replica_trace("after e2e loop")
    e2e["full_frames"] = (eng.delta_full_frames - ff0) / max(W + K, 1)
    e2e["redos"] = eng.delta_redos - rd0
    e2e["delta"] = bool(G > 1 and eng.delta_upload)

    # ---- second headline metric: GAE microseconds per rollout (T x N per GPU), kernel time via CUDA-graph
    #      replays of 20 back-to-back launches (no launch gaps), plus the reference loop with torch ops on the GPU
    def gae_us(mode):
        fn = lambda: ops.gae(eng.rewards, eng.values, eng.dones, eng.next_value, eng.next_done, args.gamma,
                             args.gae_lambda, mode=mode, out=(eng.advantages, eng.returns))
        fn(); torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(20):
                fn()
        ts = []
        for _ in range(10):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); g.replay(); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3 / 20)
        return float(np.median(ts))

    def gae_ref_us():
        r, v, d, nv, nd = eng.rewards, eng.values, eng.dones, eng.next_value.view(1, -1), eng.next_done
        ts = []
        for _ in range(3):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            adv = torch.zeros_like(r); last = 0
            for t in reversed(range(T)):
                nnt = 1.0 - (nd if t == T - 1 else d[t + 1]); nvs = nv if t == T - 1 else v[t + 1]
                delta = r[t] + args.gamma * nvs * nnt - v[t]
                adv[t] = last = delta + args.gamma * args.gae_lambda * nnt * last
            b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
        return float(np.median(ts))

    gae = {"T": T, "N": N, "sequential_bit_exact_us": round(gae_us(0), 2), "chunked_scan_us": round(gae_us(1), 2),
           "reference_torch_loop_on_gpu_us": round(gae_ref_us(), 1), "algorithmic_bytes": 20 * T * N + 8 * N}

    # data-parallel correctness, checked on the hardware the number was measured on: after K + W iterations x 16
    # updates x 2 loops every rank must hold bit-identical parameters and Adam state (the reference's own cross-rank
    # check is the debug print of ppo_atari_multigpu.py:284-286)
    replicas_identical = None
    if world > 1:
        ok = torch.ones(1, device=device)
        for buf in (eng.flat.flat, eng.flat.exp_avg, eng.flat.exp_avg_sq):
            ref = buf.clone()
            dist.broadcast(ref, 0)
            if not torch.equal(ref, buf):
                ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        replicas_identical = bool(ok.item() == 1.0)

    def shutdown():
        if world > 1:
            eng._upd_graphs.clear()                # graphs that captured NCCL kernels must be gone before the communicator
            torch.cuda.synchronize()
            dist.barrier()
            dist.destroy_process_group()

    if rank != 0:
        shutdown()
        return
    steps_total = N * T * world
    sps = steps_total * K / (res["ms"] * 1e-3)
    sps_e2e = steps_total * K / (e2e["ms"] * 1e-3)
    peak_tf, peak_hbm, which = measured_peaks()
    # dominant kernel family by device time inside the timed region
    prof = sorted(res["prof"], key=lambda r: -r["ms"])
    tot_ms = sum(r["ms"] for r in prof) or 1.0
    top = next((r for r in prof if r["flops"] > 0), prof[0])
    # which roof bounds the dominant kernel: its arithmetic intensity (algorithmic flops / algorithmic bytes)
    # against the ridge of the measured peaks
    ridge = peak_tf * 1e12 / (peak_hbm * 1e9)
    intensity = top["flops"] / top["bytes"] if top["bytes"] > 0 else float("inf")
    hbm_bound = top["flops"] == 0 or intensity < ridge
    secs = top["ms"] * 1e-3
    ach_tf = top["flops"] / secs / 1e12 if secs > 0 else 0.0
    ach_gb = top["bytes"] / secs / 1e9 if secs > 0 else 0.0
    traffic = None
    for name in ("r2_traffic.json", "r1_traffic.json"):      # the newest ncu --set full capture that has this kernel
        tp = ROOT / "profiles" / name
        tr = json.loads(tp.read_text()).get(top["name"]) if tp.exists() else None
        if tr:
            traffic = {"dram_bytes_per_launch": tr["dram_bytes"], "algorithmic_bytes_per_launch": tr["algorithmic_bytes"],
                       "at_n": tr["n"], "from": f"profiles/{name} (ncu --set full)"}
            break
    roofline = {
        "bound": "hbm" if hbm_bound else "tensor", "kernel": top["name"],
        "achieved": round(ach_gb if hbm_bound else ach_tf, 2), "peak": peak_hbm if hbm_bound else peak_tf,
        "unit": "GB/s" if hbm_bound else "TFLOP/s",
        "frac": round(ach_gb / peak_hbm if hbm_bound else ach_tf / peak_tf, 4), "traffic": traffic,
        "peak_source": f"{which} " + ("hbm_gbps" if hbm_bound else "bf16_tflops_sustained"),
        "arithmetic_intensity_flop_per_byte": round(intensity, 1), "ridge_flop_per_byte": round(ridge, 1),
        "achieved_tflops": round(ach_tf, 2), "achieved_gbs": round(ach_gb, 1),
        "share_of_kernel_time": round(top["ms"] / tot_ms, 4), "launches": top["launches"],
        "avg_launch_us": round(1e3 * top["ms"] / max(top["launches"], 1), 2),
        "job_tensor_frac": round(sps / world * FLOP_PER_ENV_STEP / (peak_tf * 1e12), 4),
        "job_hbm_frac": round(sps / world * HBM_BYTES_PER_ENV_STEP / (peak_hbm * 1e9), 4),
        "kernels": [{"name": r["name"], "ms_per_step": round(r["ms"] / K, 4), "launches_per_step": r["launches"] // K,
                     "tflops": round(r["flops"] / (r["ms"] * 1e-3) / 1e12, 2) if r["ms"] > 0 and r["flops"] > 0 else None,
                     "gbs": round(r["bytes"] / (r["ms"] * 1e-3) / 1e9, 1) if r["ms"] > 0 and r["bytes"] > 0 else None,
                     "hbm_frac": round(r["bytes"] / (r["ms"] * 1e-3) / 1e9 / peak_hbm, 3) if r["ms"] > 0 and r["bytes"] > 0 else None}
                    for r in prof],
    }
    out = {
        "metric": METRIC, "value": round(sps, 1), "unit": "env_steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": round(res["ms"] / K, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": opt.precision, "data": "synthetic",
        "config": bench_config(N, T, world),
        "clocks": res["clocks"],
        "e2e": {"value": round(sps_e2e, 1), "unit": "env_steps/s", "ms_per_step": round(e2e["ms"] / K, 3),
                "h2d_bytes_per_step": int(e2e["h2d"]), "d2h_bytes_per_step": int(e2e["d2h"]), "clocks": e2e["clocks"],
                "rollout_ms": round(e2e.get("rollout_ms", 0.0), 3), "update_ms": round(e2e.get("update_ms", 0.0), 3),
                "h2d_gbps_during_rollout": round(e2e["h2d"] / max(e2e.get("rollout_ms", 0.0), 1e-9) * 1e-6, 1),
                "env_groups": G, "loop": "PPOEngine.collect (pipelined env groups)" if G > 1 else "policy_step / env.step",
                "host": {"cores": os.cpu_count(), "process_pinned_to_gpu_local_cores": pinned_cores,
                         "verification_threads_per_group": (eng._delta[0]["tr"].threads if getattr(eng, "_delta", None) else 0)},
                **({"host_us_per_env_step": e2e["host_us_per_env_step"]} if "host_us_per_env_step" in e2e else {}),
                "observations": ("frame-stacked synthetic env (envpool stack_num=4 semantics)" if obs_mode == "stack" and G > 1
                                 else "unrelated random batches"),
                "upload": ({"mode": "frame-stack delta: newest plane of every env + whole observations of done envs; "
                                    "shifted-stack property verified on the host for every env, every step",
                            "whole_observations_per_iteration": round(e2e["full_frames"], 1), "redone_steps": e2e["redos"]}
                           if e2e["delta"] else {"mode": "whole observation every step"})},
        "gpu_launches": int(res["launches"]),
        "update_cuda_graphs": {"enabled": bool(eng.update_graphs and world == 1 or os.environ.get("CLEANRL_B200_UPDATE_GRAPHS_DP", "0") == "1"),
                               "ms_per_step_eager_with_profile_events": round(res["eager_ms"] / K, 3)},
        "gae_us_per_rollout": gae,
        "roofline": roofline,
        "losses_last": {k: (float(v) if isinstance(v, (int, float)) else None) for k, v in (e2e["stats"] or {}).items()
                        if k in ("pg_loss", "v_loss", "entropy", "approx_kl")},
    }
    if e2e_whole is not None:
        out["e2e_whole_upload"] = {
            "value": round(steps_total * K / (e2e_whole["ms"] * 1e-3), 1), "unit": "env_steps/s",
            "ms_per_step": round(e2e_whole["ms"] / K, 3), "h2d_bytes_per_step": int(e2e_whole["h2d"]),
            "d2h_bytes_per_step": int(e2e_whole["d2h"]), "rollout_ms": round(e2e_whole.get("rollout_ms", 0.0), 3),
            "update_ms": round(e2e_whole.get("update_ms", 0.0), 3), "observations": "unrelated random batches, uploaded whole"}
    if world > 1:
        out["replicas_identical"] = replicas_identical
        out["exchange"] = {"collectives_per_update": 2 if eng.overlap_exchange else 1,
                           "overlapped_with_backward": bool(eng.overlap_exchange), "bytes_per_update": eng.flat.flat.numel() * 4}
    if world == 1 and not opt.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(opt)
    if world == 1 and not opt.no_gpu_eager_baseline:
        out["gpu_eager_baseline"] = gpu_eager_baseline(opt)
    if world == 1 and not opt.no_extra:
        del eng
        torch.cuda.empty_cache()
        out["extra"] = extra_configs()
    print(json.dumps(out), flush=True)
    shutdown()


# ------------------------------------------------------------------ BASELINE.json configs[3] and configs[4]
def extra_configs():
    """Short measured lines for the two other GPU configurations BASELINE.json names (not the headline metric):
    configs[3] ppo_continuous_action HalfCheetah-shaped, num_envs=512 (the drop-in script end to end, host envs);
    configs[4] dqn_atari replay-ring sample + TD update at batch 8192 (device-resident ring)."""
    import torch
    out = {}
    try:
        from cleanrl_b200 import ppo_continuous_action as pca

        class _NullWriter:
            def __init__(self, *a, **k): pass
            def add_text(self, *a, **k): pass
            def add_scalar(self, *a, **k): pass
            def close(self): pass

        n_envs, n_steps, iters = 512, 256, 4
        marks = []

        def on_iteration(it, engine, st):
            torch.cuda.synchronize()
            marks.append(time.time())

        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):
            pca.main(["--synthetic-env", "--num-envs", str(n_envs), "--num-steps", str(n_steps),
                      "--total-timesteps", str(n_envs * n_steps * iters), "--seed", "1"],
                     writer_factory=_NullWriter, on_iteration=on_iteration)
        sec = (marks[-1] - marks[0]) / (len(marks) - 1)
        out["config4_ppo_continuous_action"] = {
            "value": round(n_envs * n_steps / sec, 1), "unit": "env_steps/s", "ms_per_iteration": round(1e3 * sec, 2),
            "workload": f"cleanrl_b200/ppo_continuous_action.py (public script, host synthetic HalfCheetah-shaped env, obs 17 / act 6), "
                        f"num_envs={n_envs} num_steps={n_steps}, 10 epochs x 32 minibatches, fp32 kernels; {iters - 1} timed iterations "
                        "after 1 warm-up, wall clock around the whole iteration"}
    except Exception as e:  # an extra line must never take the headline down with it
        out["config4_ppo_continuous_action"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    try:
        from cleanrl_b200.agents import QNetworkAgent, dqn_update
        from cleanrl_b200.replay import DeviceReplayRing
        from cleanrl_b200.synthetic_envs import Box, Discrete

        class E:
            single_observation_space = Box(0, 255, (4, 84, 84), np.uint8)
            single_action_space = Discrete(4)

        dev = torch.device("cuda", torch.cuda.current_device())
        B, SIZE, reps = 8192, 65536, 20
        q, t = QNetworkAgent(E()).to(dev), QNetworkAgent(E()).to(dev)
        q.precision = t.precision = "bf16"
        t.load_state_dict(q.state_dict())
        ring = DeviceReplayRing(SIZE, (4, 84, 84), 1, dev)
        ring.observations.random_(0, 256)
        ring.actions.random_(0, 4); ring.rewards.normal_(); ring.dones.bernoulli_(0.02)
        ring.pos, ring.full = 0, True
        stats = torch.zeros(2, device=dev)
        for _ in range(3):
            dqn_update(q, t, ring, ring.sample(B), 0.99, 1e-4, huber=True, stats=stats)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            dqn_update(q, t, ring, ring.sample(B), 0.99, 1e-4, huber=True, stats=stats)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / reps
        out["config5_dqn_atari"] = {
            "value": round(B / (ms * 1e-3), 1), "unit": "transitions/s", "ms_per_sample_plus_update": round(ms, 3),
            "workload": f"replay-ring sample + Huber TD update, batch {B}, ring of {SIZE} uint8 frames resident in HBM, "
                        f"bf16 tensor-core QNetwork; {reps} timed updates (CUDA events) after 3 warm-up"}
        del q, t, ring
        torch.cuda.empty_cache()
    except Exception as e:
        out["config5_dqn_atari"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    return out


# ---------------------------------------------------------------------- reference / cpu legs
def cpu_sample(opt, n_slices, warmup_slices, threads):
    """oracle/ppo_port.run_sliced: 1/16-iteration slices of the reference's torch-CPU loop at FULL tensor shapes
    (num_envs x num_steps rollout buffer, full minibatch size); 16 slices = one iteration's work."""
    from oracle import ppo_port
    return ppo_port.run_sliced(num_envs=opt.num_envs, num_steps=opt.num_steps, slices_per_iteration=16, n_slices=n_slices,
                               warmup_slices=warmup_slices, seed=1, threads=threads)


def cpu_baseline(opt):
    """The reference loop (oracle port, validated against the unmodified script) on the host cores, bounded sample:
    2 timed slices (after 1 warm-up slice) of 1/16 iteration each, all tensors at the benchmarked shapes."""
    import torch
    cores = os.cpu_count() or 1
    threads = min(cores, 64)
    r = cpu_sample(opt, 2, 1, threads)
    secs = sum(r["slice_seconds"])
    steps = r["env_steps_per_slice"] * len(r["slice_seconds"])
    return {"value": round(steps / secs, 1), "unit": "env_steps/s", "cores": threads, "kind": "port",
            "sample": f"{len(r['slice_seconds'])} slices of 1/16 PPO iteration at num_envs={opt.num_envs}, num_steps={opt.num_steps}, "
                      f"minibatch {r['minibatch_size']} (full shapes): {steps} env steps in {secs:.1f} s, "
                      f"torch {torch.__version__} CPU, {threads} threads of {cores} host cores"}


def gpu_eager_baseline(opt):
    """SURVEY 8(d)(ii): what `python cleanrl/ppo_atari_envpool.py --cuda` executes on this same GPU -- fp32 rollout
    storage on the device, eager torch / cuDNN / cuBLAS ops, autograd, foreach Adam, per-step action sync -- restated
    by oracle/ppo_port.py with device="cuda" (no /root/reference on the GPU box).  2 iterations, the second is timed."""
    import torch
    from oracle import ppo_port
    try:
        r = ppo_port.run(num_envs=opt.num_envs, num_steps=opt.num_steps, num_iterations=2, seed=1, env_mode="pool",
                         device="cuda", total_iterations=10)
        sec = r["iter_seconds"][-1]
        out = {"value": round(opt.num_envs * opt.num_steps / sec, 1), "unit": "env_steps/s", "kind": "port on cuda (torch eager)",
               "iter_seconds": [round(x, 3) for x in r["iter_seconds"]], "torch": torch.__version__}
    except Exception as e:  # the baseline must never take the product's number down with it
        out = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    torch.cuda.empty_cache()
    return out


def run_reference(opt):
    """--impl reference: the reference's own CPU implementation of the path (torch CPU loop, all host threads it can
    use) -- the oracle port, because /root/reference does not exist on the GPU box.  Same `config` as our arm; every
    step is a bounded sample of that workload: one 1/16-iteration slice at full tensor shapes (see cpu_sample)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    threads = min(cores, 64)
    K, W = opt.steps, opt.warmup
    r = cpu_sample(opt, K, W, threads)
    secs = sum(r["slice_seconds"])
    steps = r["env_steps_per_slice"] * K
    sps = steps / secs
    sample = (f"each step = one slice of 1/16 PPO iteration at full shapes (num_envs={opt.num_envs}, num_steps={opt.num_steps}, "
              f"minibatch {r['minibatch_size']}): {opt.num_steps // 16} policy steps x {opt.num_envs} envs + 1 minibatch update; "
              f"{K} timed + {W} warm-up slices, torch {torch.__version__} CPU, {threads} threads of {cores} host cores")
    line = {
        "impl": "reference", "metric": METRIC, "value": round(sps, 1), "unit": "env_steps/s", "n_gpus": opt.gpus,
        "steps": K, "warmup": W, "ms_per_step": round(1e3 * secs / K, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(opt.num_envs, opt.num_steps, opt.gpus),
        "cpu_baseline": {"value": round(sps, 1), "unit": "env_steps/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": round(sps, 1), "unit": "env_steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--num-envs", type=int, default=1024)
    ap.add_argument("--num-steps", type=int, default=128)
    ap.add_argument("--precision", choices=["bf16", "fp32"], default="bf16")
    ap.add_argument("--env-groups", type=int, default=2)
    ap.add_argument("--env-obs", choices=["stack", "pool"], default="stack")
    ap.add_argument("--no-whole-upload-arm", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of `value`, write what its last step computed to DIR/<name>.npy")
    opt = ap.parse_args()
    if opt.impl == "reference":
        run_reference(opt)
    else:
        run_ours(opt)


if __name__ == "__main__":
    main()
