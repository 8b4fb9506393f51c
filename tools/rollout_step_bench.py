"""Rollout policy step: the launch chain (frames_to_s2d_u8 + NatureCNNBf16.forward + categorical_sample) against the one-call
step (b200rl_naturecnn_bf16_rollout_step: conv tower + fc + heads/sampler), timed in the same process, alternating.

For each batch size n (1024 = bench.py's num_envs, 512 = one of two env groups, 160 = a chunk) both variants are captured as a
CUDA graph of 128 steps that write into the engine's own [T, N, ...] rollout storage from a device-resident frame pool (as
bench.py's `value` does, so the slot writes stream to HBM); each graph is replayed --reps times, alternating, and the median
device time per step is reported.  An eager pass with b200rl_profile_* gives the per-kernel table.  One JSON line on stdout
(and in --out), with the device name, power limit and SM clock read by nvidia-smi in the same run.

    python tools/rollout_step_bench.py [--reps 20] [--out FILE]
"""
import argparse
import ctypes
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from bench import ppo_args  # noqa: E402
from cleanrl_b200 import _lib, build  # noqa: E402
from cleanrl_b200.agents import NatureCNNAgent  # noqa: E402
from cleanrl_b200.ppo_engine import PPOEngine  # noqa: E402
from cleanrl_b200.synthetic_envs import SyntheticAtariVec  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, sm, smmax = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": plim, "clocks_sm": sm, "clocks_max_sm": smmax}
    except Exception as e:                      # the timing itself needs no nvidia-smi
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--sizes", default="1024,512,160")
    ap.add_argument("--out", default=None)
    opt = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("rollout_step_bench.py needs a CUDA device")
    build.build()
    lib = _lib.load()
    N, T = 1024, 128
    dev = torch.device("cuda:0")
    np.random.seed(1); torch.manual_seed(1)
    envs = SyntheticAtariVec(N, seed=1, mode="pool", pinned=True)
    envs.single_observation_space, envs.single_action_space = envs.observation_space, envs.action_space
    agent = NatureCNNAgent(envs).to(dev)
    agent.precision = "bf16"
    eng = PPOEngine(agent, ppo_args(N, T, 4, "bf16"), (4, 84, 84), np.uint8, N, dev, gae_mode=1)
    assert eng.u8_rollout and eng._fused_rollout()
    pool = torch.from_numpy(envs._batches).to(dev)
    P = pool.shape[0]
    agent._tc_plan()

    def chain(step, n):
        sl = slice(0, n)
        eng._to_storage(pool[step % P][:n], step, sl)
        agent.sample_into(eng.obs[step][sl], eng.actions[step][sl], eng.logprobs[step][sl], eng.values[step][sl])

    def fused(step, n):
        eng._rollout_step(step, pool[step % P][:n], slice(0, n))

    variants = {"chain": chain, "fused": fused}
    result = {"gpu": gpu_info(), "T": T, "reps": opt.reps, "sizes": {}}
    for n in [int(x) for x in opt.sizes.split(",")]:
        graphs = {}
        for name, fn in variants.items():
            rng = torch.cuda.get_rng_state(dev)
            for step in range(T):                  # eager warm-up: workspaces, tensor maps, smem opt-ins
                fn(step, n)
            torch.cuda.synchronize()
            torch.cuda.set_rng_state(rng, dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for step in range(T):
                    fn(step, n)
            graphs[name] = g
        times = {k: [] for k in graphs}
        for _ in range(2):
            for g in graphs.values():
                g.replay()
        for _ in range(opt.reps):
            for name, g in graphs.items():        # alternating
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); g.replay(); e1.record()
                e1.synchronize()
                times[name].append(e0.elapsed_time(e1) * 1e3 / T)
        row = {k: {"median_us_per_step": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}
               for k, v in times.items()}
        row["speedup"] = row["chain"]["median_us_per_step"] / row["fused"]["median_us_per_step"]
        # per-kernel table: an eager pass of 16 steps per variant with CUDA-event brackets
        for name, fn in variants.items():
            lib.b200rl_profile_reset()
            lib.b200rl_profile_enable(1)
            for step in range(16):
                fn(step, n)
            torch.cuda.synchronize()
            lib.b200rl_profile_enable(0)
            buf = ctypes.create_string_buffer(1 << 16)
            _lib.check(lib.b200rl_profile_summary(buf, 1 << 16), "profile_summary")
            row[name]["eager_profile_16_steps"] = json.loads(buf.value.decode())
        result["sizes"][str(n)] = row
        del graphs
    line = json.dumps(result)
    print(line)
    if opt.out:
        Path(opt.out).parent.mkdir(parents=True, exist_ok=True)
        Path(opt.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
