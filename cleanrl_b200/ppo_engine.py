"""B200-native PPO iteration engine: rollout storage, policy step, GAE, minibatch update.

This is the loop body of the reference scripts (cleanrl/ppo.py:185-310 and its
twins in ppo_atari_envpool.py / ppo_atari_multigpu.py) re-designed around
device-resident buffers and fused kernels:

* observations cross PCIe as uint8: pinned host batch -> async H2D in chunks on a
  copy stream while the compute stream already converts / evaluates the chunks
  that have landed; the rollout slot ``obs[t]`` holds them as space-to-depth bf16
  (tensor-core path, converted once per env step) or uint8 (exact fp32 path).
  The reference converts to fp32 on the host and keeps a 14.8 GB fp32 buffer
  (ppo_atari_envpool.py:203,239);
* rewards / dones are kept in pinned host memory during the rollout and
  uploaded once per iteration (the reference does 2 H2D + N scalar syncs per step);
* one launch per network layer + one sampler launch per env step, replayed as a
  CUDA graph per rollout slot, no autograd;
* GAE is one kernel; the loss (+its gradient) is one kernel; clip+Adam is one
  fused pass over a flat parameter vector; the DP gradient exchange is ONE
  in-place all-reduce of that flat vector (ppo_atari_multigpu.py:360-374).

numpy's global RNG still drives the minibatch shuffle and torch's generator the
sampling noise, so seeds mean what they mean in the reference (ppo.py:153-157).
"""
from __future__ import annotations

import os
import time

import numpy as np
import torch

from . import ops

STAT_NAMES = ops.STAT_NAMES


def _torch_dtype(np_dtype):
    return torch.uint8 if np.dtype(np_dtype) == np.uint8 else torch.float32


def _pin(t):
    """Page-lock a host staging buffer when a CUDA runtime exists (async H2D/D2H need it)."""
    return t.pin_memory() if torch.cuda.is_available() else t


def _sync():
    if torch.cuda.is_available():
        torch.cuda.current_stream().synchronize()


class PPOEngine:
    # The product path is CUDA-only.  The CPU test-suite (tests/cpu_backend.py) flips this to drive the
    # host-side logic (sharding, seeding, flat-gradient all-reduce over gloo) with injected torch ops.
    ALLOW_NON_CUDA_FOR_TESTS = False

    def __init__(self, agent, args, obs_shape, obs_dtype, num_envs, device, world_size=1, gae_mode=0,
                 all_reduce=None, cuda_graphs=None):
        if device.type != "cuda" and not PPOEngine.ALLOW_NON_CUDA_FOR_TESTS:
            raise RuntimeError("PPOEngine drives libb200rl CUDA kernels and needs a CUDA device; "
                               "there is no CPU fallback (got device=%s)" % device)
        self.agent, self.args, self.device = agent, args, device
        self.T, self.N = int(args.num_steps), int(num_envs)
        self.B = self.T * self.N
        self.num_minibatches = int(args.num_minibatches)
        self.M = self.B // self.num_minibatches
        self.world_size = int(world_size)
        self.all_reduce = all_reduce
        self.overlap_exchange = (device.type == "cuda" and world_size > 1 and
                                 os.environ.get("CLEANRL_B200_OVERLAP_EXCHANGE", "1") != "0")
        self._xchg_stream = None
        self.gae_mode = gae_mode
        T, N = self.T, self.N
        self.obs_dtype = _torch_dtype(obs_dtype)
        f32 = torch.float32
        # bf16 tensor-core path on Atari frames: the rollout is stored ONCE as space-to-depth bf16
        # [T,N,21,21,64] (converted per env step from the uint8 staging batch); every minibatch pass
        # then gathers 128-byte pixels directly -- no per-minibatch uint8 decode, no fp32 obs.
        self.sort_minibatch = os.environ.get("CLEANRL_B200_SORT_MINIBATCH", "1") != "0"
        self.s2d = (getattr(agent, "precision", "fp32") == "bf16" and self.obs_dtype == torch.uint8
                    and tuple(obs_shape) == (4, 84, 84) and device.type == "cuda")
        # uint8 rollout (default): every frame is kept ONCE per orientation as 1-byte space-to-depth pixels --
        # row-major [T,N,441,64] for conv1's forward on the integer tensor cores, channel-major [T,N,64,448] for its weight
        # gradient -- 28 KB per frame and pass instead of 56 KB of bf16 (CLEANRL_B200_OBS_LAYOUT=bf16 keeps the old layout)
        self.obs_t = self.next_obs_t = None
        self.u8_rollout = self.s2d and os.environ.get("CLEANRL_B200_OBS_LAYOUT", "u8") != "bf16"
        if self.s2d:
            if self.u8_rollout:
                self.obs = ops.alloc_u8_rollout_rows((T, N, 441, 64), device)
                self.obs_t = torch.zeros((T, N, 64, 448), dtype=torch.uint8, device=device)
                self.next_obs_t = torch.zeros((N, 64, 448), dtype=torch.uint8, device=device)
            else:
                self.obs = torch.zeros((T, N, 21, 21, 64), dtype=torch.bfloat16, device=device)
            self.obs_u8 = torch.zeros((N,) + tuple(obs_shape), dtype=torch.uint8, device=device)
        else:
            self.obs = torch.zeros((T, N) + tuple(obs_shape), dtype=self.obs_dtype, device=device)
        self.act_dim = int(getattr(agent, "action_dim", 0))
        if self.act_dim:     # continuous actions (ppo_continuous_action.py:213): f32 [T, N, D]
            self.actions = torch.zeros((T, N, self.act_dim), dtype=f32, device=device)
        else:                # discrete: stored as int64 (the reference stores fp32 and re-casts .long() per minibatch)
            self.actions = torch.zeros((T, N), dtype=torch.int64, device=device)
        self.logprobs = torch.zeros((T, N), dtype=f32, device=device)
        self.values = torch.zeros((T, N), dtype=f32, device=device)
        self.rewards = torch.zeros((T, N), dtype=f32, device=device)
        self.dones = torch.zeros((T, N), dtype=f32, device=device)
        self.advantages = torch.zeros((T, N), dtype=f32, device=device)
        self.returns = torch.zeros((T, N), dtype=f32, device=device)
        self.next_obs = ops.alloc_u8_rollout_rows((N, 441, 64), device) if self.u8_rollout else torch.zeros_like(self.obs[0])
        self.next_done = torch.zeros(N, dtype=f32, device=device)
        self.next_value = torch.zeros(N, dtype=f32, device=device)
        # pinned host mirrors
        self.rewards_h = _pin(torch.zeros((T, N), dtype=f32))
        self.dones_h = _pin(torch.zeros((T, N), dtype=f32))
        self.next_done_h = _pin(torch.zeros(N, dtype=f32))
        self.actions_h = _pin(torch.zeros_like(self.actions[0], device="cpu"))
        self.obs_stage_h = _pin(torch.zeros((N,) + tuple(obs_shape), dtype=self.obs_dtype))
        E = int(args.update_epochs)
        self.b_inds_h = _pin(torch.zeros((E, self.B), dtype=torch.int64))   # one slot per epoch: a pinned
        self.b_inds = torch.zeros((E, self.B), dtype=torch.int64, device=device)  # source is never rewritten in flight
        n_upd = int(args.update_epochs) * self.num_minibatches
        self.stats = torch.zeros(max(n_upd, 1), 16, dtype=f32, device=device)
        self.stats_h = _pin(torch.zeros(max(n_upd, 1), 16, dtype=f32))
        self.grad_norm = torch.zeros(1, dtype=f32, device=device)
        # CUDA graphs of the update: one graph per epoch (sort + its minibatch updates), replayed every iteration; the Adam
        # scalars that depend on (step, lr) come from a small device table refreshed once per iteration.  Takes the host
        # out of the update (about 650 kernel launches per iteration): the device no longer waits on python / driver jitter.
        self.update_graphs = os.environ.get("CLEANRL_B200_UPDATE_GRAPHS", "1") != "0"
        self.host_seconds = {"shuffle": 0.0, "update_enqueue": 0.0, "update_wait": 0.0}     # host wall time, accumulated
        # np.random.shuffle restated natively (bit-exact, same generator consumption; ops.numpy_global_shuffle)
        self._shuffle = (ops.numpy_global_shuffle if device.type == "cuda" and os.environ.get("CLEANRL_B200_NATIVE_SHUFFLE", "1") != "0"
                         else np.random.shuffle)
        self._upd_graphs, self._upd_kernels, self._upd_iters = {}, {}, 0
        self.hyper = torch.zeros(max(n_upd, 1), 2, dtype=f32, device=device)
        self.hyper_h = _pin(torch.zeros(max(n_upd, 1), 2, dtype=f32))
        self.flat = agent.flat
        if self.overlap_exchange and hasattr(agent, "grad_tail"):
            agent.grad_tail()          # create the tail event BEFORE the first backward records it
        # One CUDA graph per rollout slot: the per-step device work (frame conversion, 5 network launches, noise
        # draw, sampler) becomes a single graph launch that writes straight into obs[t]/actions[t]/...; the
        # rollout is launch-latency bound otherwise (~12 launches + torch ops per 1024-env step).
        if cuda_graphs is None:
            cuda_graphs = os.environ.get("CLEANRL_B200_CUDA_GRAPHS", "1") != "0"
        self.cuda_graphs = bool(cuda_graphs) and device.type == "cuda"
        # e2e pipeline: the pinned batch goes up in H2D_CHUNKS pieces on a copy stream while the compute stream
        # already converts / evaluates the pieces that have landed (PCIe is the longest stage of a step)
        chunks = int(os.environ.get("CLEANRL_B200_H2D_CHUNKS", "4"))
        self.h2d_chunks = chunks if (self.cuda_graphs and getattr(self, "s2d", False) and chunks > 1
                                     and N % chunks == 0 and N // chunks >= 128) else 1
        # chunk sizes: a short LAST chunk keeps the work that cannot overlap the upload (its conversion + forward,
        # the sampler, the action D2H) small; every chunk's compute is still shorter than the next chunk's upload
        C = self.h2d_chunks
        if C == 4 and N % 16 == 0:
            sizes = [5 * N // 16, 5 * N // 16, 4 * N // 16, 2 * N // 16]
        else:
            sizes = [N // C] * C
        self.chunk_bounds = [(sum(sizes[:c]), sum(sizes[:c + 1])) for c in range(C)]
        self.noise_buf = None
        if self.h2d_chunks > 1:
            self.copy_stream = torch.cuda.Stream(device=device)
            self.chunk_events = [torch.cuda.Event() for _ in range(self.h2d_chunks)]
            self.noise_buf = torch.zeros(agent.noise_shape(N), dtype=f32, device=device)
        self._parts = None
        # frame-stack delta upload (grouped loop, uint8 rollout): only the newest frame plane of every env crosses PCIe, the
        # device rebuilds slot t from slot t-1, a host worker pool verifies the shifted-stack property (csrc/frame_stack.cu)
        # Default: on for a single process per host, off when several ranks share the host (LOCAL_WORLD_SIZE > 1): the
        # verification and the leaner launch path make the rollout HOST-bound instead of PCIe-bound, which wins on an idle host
        # (1.39 M vs 1.03 M env-steps/s) and loses when the ranks' worker pools compete for the same cores and memory
        # bandwidth (profiles/r2_host_sensitivity.md).  CLEANRL_B200_DELTA_UPLOAD=1 / 0 overrides either way.
        want_delta = os.environ.get("CLEANRL_B200_DELTA_UPLOAD")
        if want_delta is None:
            want_delta = "1" if int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1) <= 1 else "0"
        self.delta_upload = bool(getattr(self, "u8_rollout", False)) and want_delta != "0"
        self._delta_allowed = self.delta_upload      # trackers / staging exist; ``delta_upload`` is the current state
        self._delta = None
        self.delta_redos = 0             # steps redone because an env broke the shifted-stack contract without being done
        self.delta_full_frames = 0       # env observations uploaded whole (resets, first step, redos)
        self._graphs = {}
        self._graph_pool = None
        self._graph_kernels = {}
        self._graph_warm = set()
        self.graph_launches = 0          # libb200rl kernels executed through graph replays
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        self.kernel_launches = 0

    # ------------------------------------------------------------------ rollout
    def _to_storage(self, src_u8, step, sl=slice(None)):
        """uint8 NCHW frames (device) -> the rollout slot ``step`` (None = the bootstrap slot ``next_obs``), rows ``sl``."""
        dst = self.next_obs if step is None else self.obs[step]
        if self.u8_rollout:
            dst_t = self.next_obs_t if step is None else self.obs_t[step]
            ops.frames_to_s2d_u8(src_u8, dst[sl], dst_t[sl])
        else:
            ops.frames_to_s2d(src_u8, out=dst[sl])

    def _upload_obs(self, step, obs_np, convert=True):
        """Host frames -> device (pinned staging when needed) -> rollout slot ``step`` (None = bootstrap slot)."""
        dst = self.next_obs if step is None else self.obs[step]
        src = torch.from_numpy(np.ascontiguousarray(obs_np))
        if src.dtype != self.obs_dtype:
            src = src.to(self.obs_dtype)
        if not src.is_pinned():
            self.obs_stage_h.copy_(src)
            src = self.obs_stage_h
        if self.s2d:
            self.obs_u8.copy_(src, non_blocking=True)
            if convert:
                self._to_storage(self.obs_u8, step)
        else:
            dst.copy_(src, non_blocking=True)
        self.h2d_bytes += src.numel() * src.element_size()

    def _fused_rollout(self):
        """uint8 rollout layout with an agent that has the one-call rollout step (conv tower + fc + heads/sampler)."""
        return self.u8_rollout and getattr(self.agent, "precision", "fp32") == "bf16" and hasattr(self.agent, "rollout_step_into")

    def _rollout_step(self, step, src_u8, sl=slice(None), noise=None):
        """Policy step of rows ``sl`` of slot ``step``: ``src_u8`` = their uint8 NCHW frames (None: the slot already holds
        them).  One native call on the u8 rollout layout; otherwise storage conversion, then forward + sampler."""
        if self._fused_rollout():
            self.agent.rollout_step_into(src_u8, self.obs[step][sl], self.obs_t[step][sl], self.actions[step][sl],
                                         self.logprobs[step][sl], self.values[step][sl], noise=noise)
            return
        if src_u8 is not None:
            self._to_storage(src_u8, step, sl)
        self.agent.sample_into(self.obs[step][sl], self.actions[step][sl], self.logprobs[step][sl], self.values[step][sl],
                               noise=noise)

    def _step_device_work(self, step, noise=None):
        """Everything a policy step does on the device after the observation batch has landed."""
        if self.s2d:
            return self._rollout_step(step, self.obs_u8, noise=noise)
        self.agent.sample_into(self.obs[step], self.actions[step], self.logprobs[step], self.values[step], noise=noise)

    def _chunk_device_work(self, step, c):
        sl = slice(*self.chunk_bounds[c])
        self._rollout_step(step, self.obs_u8[sl], sl, noise=self.noise_buf[sl])

    def _run_step(self, step, chunk=None):
        if chunk is not None:
            work, key = (lambda: self._chunk_device_work(step, chunk)), (step, chunk)
            return self._run_graphed(work, key, warm_key=("c", chunk))
        if self._graphable() and not getattr(self.agent.noise_fn, "graph_safe", False):
            # the noise source cannot be captured (e.g. a CPU generator injected by the parity tests): draw the
            # step's noise eagerly -- ONE draw per step, as the reference -- and let the graph consume the buffer
            if self.noise_buf is None:
                self.noise_buf = torch.zeros(self.agent.noise_shape(self.N), dtype=torch.float32, device=self.device)
            self.agent.draw_noise_into(self.noise_buf)
            return self._run_graphed(lambda: self._step_device_work(step, noise=self.noise_buf), step, warm_key=("f", 0))
        return self._run_graphed(lambda: self._step_device_work(step), step, warm_key=("f", 0))

    def _graphable(self):
        return self.cuda_graphs and getattr(self.agent, "graph_capturable", getattr(self.agent, "graph_friendly", False))

    def _run_graphed(self, work, key, warm_key):
        if not self._graphable():
            return work()
        if hasattr(self.agent, "_tc_plan") and getattr(self.agent, "precision", "fp32") == "bf16":
            self.agent._tc_plan()                      # (re)pack weights outside the graph
        g = self._graphs.get(key)
        if g is None:
            if warm_key not in self._graph_warm:       # allocate workspaces once (eager), then capture
                rng = torch.cuda.get_rng_state(self.device)     # the warm-up must not consume sampling noise
                work()
                torch.cuda.current_stream().synchronize()
                torch.cuda.set_rng_state(rng, self.device)
                self._graph_warm.add(warm_key)
            from . import _lib
            l0 = _lib.load().b200rl_launch_count()
            g = torch.cuda.CUDAGraph()
            if self._graph_pool is None:
                self._graph_pool = torch.cuda.graph_pool_handle()      # one private pool shared by all step graphs
            with torch.cuda.graph(g, pool=self._graph_pool):
                work()
            self._graphs[key] = g
            if hasattr(self.agent, "pin_workspaces"):
                self.agent.pin_workspaces()     # captured graphs hold raw pointers into the activation workspaces
            self._graph_kernels[key] = _lib.load().b200rl_launch_count() - l0
        g.replay()
        self.graph_launches += self._graph_kernels[key]

    @torch.no_grad()
    def policy_step(self, step, next_obs_np, next_done_np):
        """obs[step] <- next_obs (H2D), sample actions, return them as a host int64 array.
        Reference: ppo.py:194-205 (store obs/done, no-grad policy, action.cpu())."""
        if self.h2d_chunks > 1 and self._graphable():
            self._pipelined_step(step, next_obs_np)        # the upload is the critical path: enqueue it first
            self.dones_h[step].copy_(torch.as_tensor(np.asarray(next_done_np, dtype=np.float32)))
        else:
            self.dones_h[step].copy_(torch.as_tensor(np.asarray(next_done_np, dtype=np.float32)))
            self._upload_obs(step, next_obs_np, convert=False)
            self._run_step(step)
        self.actions_h.copy_(self.actions[step], non_blocking=True)
        self.d2h_bytes += self.actions_h.numel() * self.actions_h.element_size()
        _sync()
        return self.actions_h.numpy()

    def _pipelined_step(self, step, obs_np):
        """H2D of chunk c+1 overlaps frame conversion + policy of chunk c (separate copy stream + events); the
        step's sampling noise is ONE draw for the whole batch, as in the unchunked path and the reference."""
        src = torch.from_numpy(np.ascontiguousarray(obs_np))
        if not src.is_pinned():
            self.obs_stage_h.copy_(src)
            src = self.obs_stage_h
        C = self.h2d_chunks
        main = torch.cuda.current_stream()
        with torch.cuda.stream(self.copy_stream):
            for c, (lo, hi) in enumerate(self.chunk_bounds):
                self.obs_u8[lo:hi].copy_(src[lo:hi], non_blocking=True)
                self.chunk_events[c].record(self.copy_stream)
        self.h2d_bytes += src.numel()
        self.agent.draw_noise_into(self.noise_buf)
        for c in range(C):
            main.wait_event(self.chunk_events[c])
            self._run_step(step, chunk=c)

    @torch.no_grad()
    def policy_step_resident(self, step, obs_dev, done_dev=None):
        """Device-resident variant (inputs already in HBM, no host round trip): used to measure the
        kernel-side throughput of the rollout step; actions stay on the device."""
        if self.s2d and obs_dev.dtype == torch.uint8:
            self.obs_u8.copy_(obs_dev)
        else:
            self.obs[step].copy_(obs_dev)
        self._run_step(step)

    @torch.no_grad()
    def rollout_resident(self, obs_pool):
        """All T policy steps over device-resident frame batches ``obs_pool[t % P]`` (uint8 [P,N,4,84,84] or the
        engine's storage dtype) replayed as ONE CUDA graph: the kernel-side throughput of the rollout without a
        host launch per step (measurement path of bench.py's ``value``; the public loop is ``policy_step``)."""
        P = obs_pool.shape[0]

        def work():
            for step in range(self.T):
                src = obs_pool[step % P]
                if self.s2d and src.dtype == torch.uint8:
                    self._rollout_step(step, src)
                    continue
                self.obs[step].copy_(src)
                self.agent.sample_into(self.obs[step], self.actions[step], self.logprobs[step], self.values[step])

        if not getattr(self.agent, "graph_friendly", False):
            return work()          # the noise draw cannot be captured: plain launches
        self._run_graphed(work, ("rollout", obs_pool.data_ptr(), P), warm_key="r")

    # ------------------------------------------------------------ pipelined rollout over env groups
    # The reference steps all envs, then runs the policy on all envs (ppo_atari_envpool.py:224-247): host and device take
    # turns, and PCIe idles while the last chunk is evaluated, the actions come back and the env steps.  With the envs in P
    # independent groups (each its own vector env over a contiguous slice of the N envs) group B's frames cross PCIe while
    # group A is evaluated, its actions return and its env steps; A's next frames queue behind B's.  Per env nothing changes:
    # same policy, same per-step noise tensor (ONE draw per step for all N envs, the reference's RNG contract), same buffers.
    def _part_setup(self, P):
        if getattr(self, "_parts", None) is not None and len(self._parts) == P:
            return
        N = self.N
        assert N % P == 0, "num_envs must be divisible by the number of env groups"
        n = N // P
        self._parts = [(p * n, (p + 1) * n) for p in range(P)]
        C = 2 if (n % 2 == 0 and n // 2 >= 64 and self.s2d and self._graphable()) else 1
        want = os.environ.get("CLEANRL_B200_PART_CHUNKS")          # upload / compute overlap granularity inside a group
        if want and self.s2d and self._graphable() and 1 <= int(want) <= 4 and n % int(want) == 0:
            C = int(want)
        self._part_chunks = [[(lo + c * (n // C), lo + (c + 1) * (n // C)) for c in range(C)] for lo, hi in self._parts]
        if getattr(self, "copy_stream", None) is None:
            self.copy_stream = torch.cuda.Stream(device=self.device)
        self._part_h2d = [[torch.cuda.Event() for _ in ch] for ch in self._part_chunks]
        self._part_d2h = [torch.cuda.Event() for _ in range(P)]
        if self.noise_buf is None:
            self.noise_buf = torch.zeros(self.agent.noise_shape(N), dtype=torch.float32, device=self.device)
        if not hasattr(self, "obs_u8"):
            self.obs_u8 = None
        self._noise_bufs = [self.noise_buf, torch.zeros_like(self.noise_buf)]      # by step parity (see _redo_part)
        self._noise_step = -1
        self._actions_np = self.actions_h.numpy()
        self._rewards_np, self._dones_np = self.rewards_h.numpy(), self.dones_h.numpy()
        self._dones_ptr = self.dones_h.data_ptr()
        self._part_d2h_bytes = n * self.actions_h.element_size() * max(1, self.act_dim)
        self._part_d2h_handles = [None] * P
        self._plans, self._plan_refs, self._plan_kernels, self._plan_stream = {}, {}, {}, None
        if self.device.type == "cuda":
            from . import _lib
            self._lib = _lib.load()
        self._delta = None
        if self._delta_allowed and self._graphable():
            u8 = torch.uint8
            self._delta = [dict(tr=ops.StackDeltaTracker(n), full_d=torch.zeros((n, 28224), dtype=u8, device=self.device),
                                last=None, boot_obs=None, consumed=torch.cuda.Event()) for _ in range(P)]
            self._new_d = torch.zeros((N, 7056), dtype=u8, device=self.device)
            self._slot_d = torch.zeros(N, dtype=torch.int32, device=self.device)
            self._mis_ptr = [d["tr"].mis_h.data_ptr() for d in self._delta]

    def _part_work(self, step, lo, hi):
        sl = slice(lo, hi)
        if self.s2d:
            return self._rollout_step(step, self.obs_u8[sl], sl, noise=self._noise_bufs[step & 1][sl])
        self.agent.sample_into(self.obs[step][sl], self.actions[step][sl], self.logprobs[step][sl], self.values[step][sl],
                               noise=self._noise_bufs[step & 1][sl])

    @torch.no_grad()
    def launch_part(self, step, part, obs_np, done_np):
        """Enqueue everything group ``part`` needs at ``step``: H2D of its frames (copy stream, in chunks), storage
        conversion + policy + sampler per chunk (main stream, graph replays), D2H of its actions.  Returns immediately."""
        if self._delta is not None and self.delta_upload:
            return self._launch_part_delta(step, part, obs_np, done_np)
        lo, hi = self._parts[part]
        src = torch.from_numpy(np.ascontiguousarray(obs_np))
        if src.dtype != self.obs_dtype:
            src = src.to(self.obs_dtype)
        if not src.is_pinned():
            self.obs_stage_h[lo:hi].copy_(src)
            src = self.obs_stage_h[lo:hi]
        main = torch.cuda.current_stream()
        dst = self.obs_u8 if self.s2d else self.obs[step]
        with torch.cuda.stream(self.copy_stream):
            for c, (clo, chi) in enumerate(self._part_chunks[part]):
                dst[clo:chi].copy_(src[clo - lo:chi - lo], non_blocking=True)
                self._part_h2d[part][c].record(self.copy_stream)
        self.h2d_bytes += src.numel() * src.element_size()
        self.dones_h[step][lo:hi].copy_(torch.as_tensor(np.asarray(done_np, dtype=np.float32)))
        if part == 0:
            self._ensure_noise(step)
        for c, (clo, chi) in enumerate(self._part_chunks[part]):
            main.wait_event(self._part_h2d[part][c])
            self._run_graphed(lambda: self._part_work(step, clo, chi), ("part", step, part, c), warm_key=("p", part, c))
        self.actions_h[lo:hi].copy_(self.actions[step][lo:hi], non_blocking=True)
        self._part_d2h[part].record(main)
        self.d2h_bytes += (hi - lo) * self.actions_h.element_size() * max(1, self.act_dim)

    def wait_actions(self, part):
        """Host view of group ``part``'s actions of the step launched last (blocks on that group's D2H event only)."""
        lo, hi = self._parts[part]
        if self._delta is not None:
            h = self._part_d2h_handles[part]
            if h is None:
                self._part_d2h[part].synchronize()
            self._join_part(part, h)          # one C call: event wait + verification join
        else:
            self._part_d2h[part].synchronize()
        return self._actions_np[lo:hi]

    # ---- frame-stack delta upload (csrc/frame_stack.cu): the observation of cleanrl/ppo_atari_envpool.py:185-196 is a stack
    # of the 4 newest frames, so planes 0..2 of an env's observation are planes 1..3 of its previous one unless it was reset.
    # Only the newest plane is uploaded (7 KB instead of 28 KB per env); the device rebuilds slot t from slot t-1.  Envs
    # flagged done go up whole; a host worker pool memcmp's the other envs against a private mirror while the device already
    # works, and a step whose env broke the contract without being done is redone from full frames before its actions are
    # handed out (``delta_redos``; an env that is not frame-stacked at all switches the engine back to whole uploads).
    def _ensure_noise(self, step):
        """The step's ONE noise draw for all N envs (the reference's RNG contract), into the buffer of the step's parity.
        ``collect`` calls it one step ahead, right after a step's last group was launched, so that the draw is off the
        critical path of the next step's first group; draws still happen once per step, in step order."""
        if self._noise_step != step:
            self.agent.draw_noise_into(self._noise_bufs[step & 1])
            self._noise_step = step

    def _slot_pair(self, step):
        """(row-major, channel-major) storage of rollout slot ``step``; ``T`` = the bootstrap slot."""
        return (self.next_obs, self.next_obs_t) if step == self.T else (self.obs[step], self.obs_t[step])

    def _part_work_delta(self, step, part, lo, hi, sample, reuse):
        sl = slice(lo, hi)
        dst_rm, dst_cm = self._slot_pair(step)
        if reuse:            # step 0 of an iteration: the observation is the one the bootstrap slot already holds
            dst_rm[sl].copy_(self.next_obs[sl])
            dst_cm[sl].copy_(self.next_obs_t[sl])
        else:
            prev_rm, prev_cm = self._slot_pair(self.T if step == 0 else step - 1)
            ops.frames_delta_s2d_u8(self._new_d[sl], prev_rm[sl], prev_cm[sl], dst_rm[sl], dst_cm[sl],
                                    full_slot=self._slot_d[sl], full_frames=self._delta[part]["full_d"])
        if sample:
            self._rollout_step(step, None, sl, noise=self._noise_bufs[step & 1][sl])

    @staticmethod
    def _host_pinned(arr):
        try:
            return bool(torch.from_numpy(arr).is_pinned())
        except Exception:
            return False

    def _launch_part_delta(self, step, part, obs_np, done_np, sample=True):
        """One env group's rollout step.  Steady state = ONE C call (b200rl_stackdelta_launch over a plan that was filled
        when the step's graphs were captured): classification + staging + verification start, the uploads, the chunk
        graphs, the actions D2H.  The first pass over a (step, group) takes the python path below it and captures."""
        d = self._delta[part]
        reuse = step == 0 and d["boot_obs"] is not None and d["boot_obs"] is obs_np
        d["boot_obs"] = obs_np if step == self.T else None
        plan = self._plans.get((step, part, reuse))
        if plan is None or self._plan_stream != torch.cuda.current_stream().cuda_stream:
            return self._launch_part_delta_capture(step, part, obs_np, done_np, sample, reuse)
        lo, hi = self._parts[part]
        n = hi - lo
        lib = self._lib
        obs, optr, ostride = None, None, 0
        if not reuse:
            obs = obs_np
            if type(obs) is not np.ndarray or obs.dtype != np.uint8 or obs.ndim != 4 or obs.strides[1:] != (7056, 84, 1):
                obs = np.ascontiguousarray(obs_np, dtype=np.uint8)
            optr, ostride = obs.__array_interface__["data"][0], obs.strides[0]
            if step == 0:
                lib.b200rl_stackdelta_invalidate(d["tr"]._h)     # an observation the engine has not seen before
        if sample:
            np.copyto(self._dones_np[step, lo:hi], done_np, casting="unsafe")
            dptr = self._dones_ptr + (step * self.N + lo) * 4
            if part == 0:
                self._ensure_noise(step)
        else:
            dkeep = np.ascontiguousarray(done_np, dtype=np.float32)
            dptr = dkeep.__array_interface__["data"][0]
        k = lib.b200rl_stackdelta_launch(self._plan_refs[(step, part, reuse)], optr, ostride, dptr)
        if k < 0:
            from . import _lib
            _lib.check(int(k), "stackdelta_launch")
        self.graph_launches += self._plan_kernels[(step, part, reuse)]
        if reuse:
            d["last"] = None
        else:
            self.h2d_bytes += n * (7056 + 4) + k * 28224
            self.delta_full_frames += k
            d["last"] = (step, obs, k, sample)
        if sample:
            self.d2h_bytes += self._part_d2h_bytes

    def _make_plan(self, step, part, reuse, sample):
        """Fill the B200rlPartLaunch of (step, group) once its chunk graphs exist (raw handles of torch's objects)."""
        import ctypes
        from . import _lib
        lo, hi = self._parts[part]
        d = self._delta[part]
        tr = d["tr"]
        chunks = self._part_chunks[part]
        keys = [("dpart", step, part, c, reuse) for c in range(len(chunks))]
        if any(k not in self._graphs for k in keys):
            return
        pl = _lib.PartLaunch()
        pl.tracker = None if reuse else tr._h
        pl.copy_stream = self.copy_stream.cuda_stream
        pl.main_stream = torch.cuda.current_stream().cuda_stream
        pl.consumed_event = d["consumed"].cuda_event
        pl.n, pl.nchunks = hi - lo, len(chunks)
        for c, (clo, chi) in enumerate(chunks):
            pl.chunk_lo[c], pl.chunk_hi[c] = clo - lo, chi - lo
            pl.h2d_event[c] = self._part_h2d[part][c].cuda_event
            pl.graph_exec[c] = self._graphs[keys[c]].raw_cuda_graph_exec()
        pl.new_d, pl.slot_d, pl.full_d = self._new_d[lo:hi].data_ptr(), self._slot_d[lo:hi].data_ptr(), d["full_d"].data_ptr()
        pl.new_h, pl.full_h, pl.slot_h = tr.new_h.data_ptr(), tr.full_h.data_ptr(), tr.slot_h.data_ptr()
        if sample:
            pl.actions_d, pl.actions_h = self.actions[step][lo:hi].data_ptr(), self.actions_h[lo:hi].data_ptr()
            pl.actions_bytes = self._part_d2h_bytes
            pl.d2h_event = self._part_d2h[part].cuda_event
        key = (step, part, reuse)
        self._plans[key] = pl
        self._plan_refs[key] = ctypes.byref(pl)
        self._plan_kernels[key] = sum(self._graph_kernels[k] for k in keys)
        self._plan_stream = torch.cuda.current_stream().cuda_stream      # (a c_void_p field reads back None for stream 0)
        self._part_d2h_handles[part] = self._part_d2h[part].cuda_event

    def _launch_part_delta_capture(self, step, part, obs_np, done_np, sample, reuse):
        lo, hi = self._parts[part]
        n = hi - lo
        d = self._delta[part]
        tr = d["tr"]
        main, cs = torch.cuda.current_stream(), self.copy_stream
        if reuse:
            d["last"] = None
            for c in range(len(self._part_chunks[part])):
                self._part_h2d[part][c].record(main)
        else:
            obs = np.asarray(obs_np)
            if obs.dtype != np.uint8 or obs.ndim != 4 or obs.strides[1:] != (7056, 84, 1):
                obs = np.ascontiguousarray(obs, dtype=np.uint8)
            if step == 0:
                tr.invalidate()          # an observation the engine has not seen before: every env goes up whole
            pinned = self._host_pinned(obs)
            k = tr.begin(obs, done_np, pack_new=not pinned)
            cs.wait_event(d["consumed"])                 # the staging buffers' last readers on the main stream
            if k:
                ops.h2d_rows_async(d["full_d"], tr.full_h.data_ptr(), k * 28224, k * 28224, 1, cs)
            ops.h2d_rows_async(self._slot_d[lo:hi], tr.slot_h.data_ptr(), n * 4, n * 4, 1, cs)
            if pinned:
                src, pitch = obs.__array_interface__["data"][0] + 3 * 7056, int(obs.strides[0])
            else:
                src, pitch = tr.new_h.data_ptr(), 7056
            for c, (clo, chi) in enumerate(self._part_chunks[part]):
                ops.h2d_rows_async(self._new_d[clo:chi], src + (clo - lo) * pitch, pitch, 7056, chi - clo, cs)
                self._part_h2d[part][c].record(cs)
            self.h2d_bytes += n * (7056 + 4) + k * 28224
            self.delta_full_frames += k
            d["last"] = (step, obs, k, sample)
        if sample:
            self.dones_h[step][lo:hi].copy_(torch.as_tensor(np.asarray(done_np, dtype=np.float32)))
            if part == 0:
                self._ensure_noise(step)
        for c, (clo, chi) in enumerate(self._part_chunks[part]):
            main.wait_event(self._part_h2d[part][c])
            self._run_graphed(lambda: self._part_work_delta(step, part, clo, chi, sample, reuse),
                              ("dpart", step, part, c, reuse), warm_key=("dp", part, c, sample, reuse))
        d["consumed"].record(main)
        if sample:
            self.actions_h[lo:hi].copy_(self.actions[step][lo:hi], non_blocking=True)
            self._part_d2h[part].record(main)
            self.d2h_bytes += self._part_d2h_bytes
        if os.environ.get("CLEANRL_B200_LAUNCH_PLANS", "1") != "0":
            self._make_plan(step, part, reuse, sample)

    def _join_part(self, part, d2h_event=None):
        """Join the host-side verification of the observation launched last for ``part`` (after ``d2h_event``, a raw handle,
        when given); redo the step from full frames for envs that were not a shifted stack although not done."""
        d = self._delta[part]
        tr = d["tr"]
        if d["last"] is None and d2h_event is None:
            return
        m = self._lib.b200rl_stackdelta_join(tr._h if d["last"] is not None else None, d2h_event, self._mis_ptr[part])
        tr._pending, tr._keep = False, None
        if m < 0:
            from . import _lib
            _lib.check(int(m), "stackdelta_join")
        if m > 0:
            self._redo_part(part, tr.mis_h[:int(m)].numpy().copy())
        d["last"] = None

    def _redo_part(self, part, mis):
        lo, hi = self._parts[part]
        n = hi - lo
        d = self._delta[part]
        tr = d["tr"]
        step, obs, k, sample = d["last"]
        main = torch.cuda.current_stream()
        self.copy_stream.synchronize()                   # the pinned staging buffers are about to be rewritten
        main.synchronize()
        m = len(mis)
        full = tr.full_h.numpy().reshape(n, 4, 84, 84)
        slot = tr.slot_h.numpy()
        for j, i in enumerate(mis):
            full[k + j] = obs[i]
            slot[i] = k + j
        ops.h2d_rows_async(d["full_d"][k:k + m], tr.full_h.data_ptr() + k * 28224, m * 28224, m * 28224, 1, main)
        ops.h2d_rows_async(self._slot_d[lo:hi], tr.slot_h.data_ptr(), n * 4, n * 4, 1, main)
        for clo, chi in self._part_chunks[part]:
            self._part_work_delta(step, part, clo, chi, sample, False)       # eager; same noise rows as the first attempt
        if sample:
            self.actions_h[lo:hi].copy_(self.actions[step][lo:hi], non_blocking=True)
        main.synchronize()
        self.h2d_bytes += m * 28224 + n * 4
        self.delta_full_frames += m
        self.delta_redos += 1
        if m > n // 8:
            # this env does not deliver shifted frame stacks (no frame stacking, or a different stacking order):
            # go back to whole-observation uploads for the rest of the run
            self.delta_upload = False

    def collect(self, env_parts, obs_parts, done_parts, on_step=None):
        """One rollout of T steps over ``env_parts`` (gym-0.23 style ``step(a) -> obs, reward, done, info``), software
        pipelined across the groups.  ``on_step(step, part, reward, done, info)`` sees every group step (logging).
        Returns the groups' next observations / dones for ``finish_rollout_parts`` and the next iteration."""
        P = len(env_parts)
        self._part_setup(P)
        obs_parts, done_parts = list(obs_parts), list(done_parts)
        if hasattr(self.agent, "_tc_plan") and getattr(self.agent, "precision", "fp32") == "bf16":
            self.agent._tc_plan()          # (re)pack the weights once: they do not change during a rollout
        self._noise_step = -1
        if self._delta is not None:
            for p, d in enumerate(self._delta):
                if d["last"] is not None:      # a rollout abandoned mid-step (exception in env.step): drop its pending pass
                    self._lib.b200rl_stackdelta_join(d["tr"]._h, None, self._mis_ptr[p])
                    d["tr"]._pending, d["tr"]._keep, d["last"], d["boot_obs"] = False, None, None, None
        for p in range(P):
            self.launch_part(0, p, obs_parts[p], done_parts[p])
        if self.T > 1:
            self._ensure_noise(1)
        rewards_np = self._rewards_np
        for t in range(self.T):
            for p in range(P):
                lo, hi = self._parts[p]
                action = self.wait_actions(p)
                obs, reward, done, info = env_parts[p].step(action)
                np.copyto(rewards_np[t, lo:hi], np.asarray(reward).reshape(-1), casting="unsafe")
                if on_step is not None:
                    on_step(t, p, reward, done, info)
                obs_parts[p], done_parts[p] = obs, done
                if t + 1 < self.T:
                    self.launch_part(t + 1, p, obs, done)
                    if p == P - 1 and t + 2 < self.T:
                        self._ensure_noise(t + 2)        # (its buffer was last read by step t, whose actions are all back)
        return obs_parts, done_parts

    @torch.no_grad()
    def finish_rollout_parts(self, obs_parts, done_parts):
        """``finish_rollout`` for the grouped loop: bootstrap observation / done of every group."""
        nd = np.concatenate([np.asarray(d, dtype=np.float32).reshape(-1) for d in done_parts])
        if self._delta is not None and self.delta_upload:
            for p in range(len(self._parts)):
                self._launch_part_delta(self.T, p, obs_parts[p], done_parts[p], sample=False)
            for p in range(len(self._parts)):
                self._join_part(p)
            return self.finish_rollout(None, nd, resident=False, obs_uploaded=True)   # (a redo leaves the slot correct too)
        if self.s2d:
            for (lo, hi), o in zip(self._parts, obs_parts):
                src = torch.from_numpy(np.ascontiguousarray(o))
                if not src.is_pinned():
                    self.obs_stage_h[lo:hi].copy_(src)
                    src = self.obs_stage_h[lo:hi]
                self.obs_u8[lo:hi].copy_(src, non_blocking=True)
                self.h2d_bytes += src.numel()
            self._to_storage(self.obs_u8, None)
            self.finish_rollout(None, nd, resident=False, obs_uploaded=True)
        else:
            self.finish_rollout(np.concatenate([np.asarray(o) for o in obs_parts]), nd)

    def record_reward(self, step, reward_np):
        self.rewards_h[step].copy_(torch.as_tensor(np.asarray(reward_np, dtype=np.float32).reshape(-1)))

    @torch.no_grad()
    def finish_rollout(self, next_obs_np, next_done_np, resident=False, obs_uploaded=False):
        """Bootstrap value + GAE (reference: ppo.py:217-231).  ``resident``: rewards/dones/next_obs
        were already written on the device; ``obs_uploaded``: only the bootstrap frames were."""
        if not resident:
            self.rewards.copy_(self.rewards_h, non_blocking=True)
            self.dones.copy_(self.dones_h, non_blocking=True)
            self.next_done_h.copy_(torch.as_tensor(np.asarray(next_done_np, dtype=np.float32)))
            self.next_done.copy_(self.next_done_h, non_blocking=True)
            self.h2d_bytes += 2 * self.B * 4 + self.N * 4
            if not obs_uploaded:
                self._upload_obs(None, next_obs_np)
        _, value = self.agent._forward_heads(self.next_obs)
        self.next_value.copy_(value)
        ops.gae(self.rewards, self.values, self.dones, self.next_value, self.next_done,
                self.args.gamma, self.args.gae_lambda, mode=self.gae_mode,
                out=(self.advantages, self.returns))

    # ------------------------------------------------------------------- update
    @torch.no_grad()
    def update(self, lr):
        """update_epochs x num_minibatches fused updates (reference: ppo.py:233-293).
        Returns dict of the logged scalars (last minibatch's losses, mean clipfrac)."""
        a = self.args
        B, M = self.B, self.M
        t_up = time.perf_counter()
        b_inds_np = np.arange(B)
        k = 0
        E = int(a.update_epochs)
        nmb = self.num_minibatches
        graphed = (self.update_graphs and a.target_kl is None and self._graphable() and self._upd_iters >= 1
                   and getattr(self.agent, "precision", "fp32") == "bf16" and hasattr(self.agent, "_tc_plan")
                   and (self.world_size == 1 or os.environ.get("CLEANRL_B200_UPDATE_GRAPHS_DP", "0") == "1"))
        self._upd_iters += 1
        if graphed:
            hy = self.hyper_h.numpy()
            for j in range(E * nmb):                 # the scalars of every update of this iteration (host, double, as clip_adam)
                hy[j] = ops.adam_step_scalars(self.flat.step + 1 + j, lr)
            self.hyper.copy_(self.hyper_h, non_blocking=True)
        for epoch in range(E):
            # numpy global RNG, in-place and cumulative across epochs as the reference (ppo.py:245).  A shuffle of 131 072
            # indices costs the host 1.5-3 ms: it is drawn per epoch, right before that epoch's launches, so that every
            # shuffle but the first runs while the device is still busy with the previous epoch's minibatches.
            t_sh = time.perf_counter()
            self._shuffle(b_inds_np)
            self.host_seconds["shuffle"] += time.perf_counter() - t_sh
            self.b_inds_h[epoch].copy_(torch.from_numpy(b_inds_np))        # one pinned slot per epoch: never rewritten in flight
            self.b_inds[epoch].copy_(self.b_inds_h[epoch], non_blocking=True)
            self.h2d_bytes += B * 8
            if graphed:
                g = self._upd_graphs.get(epoch)
                if g is None:
                    g = self._capture_epoch(epoch)
                g.replay()
                self.graph_launches += self._upd_kernels[epoch]
                k += nmb
                continue
            k = self._epoch_work(epoch, lr, k, False)
            if a.target_kl is not None:
                approx_kl = self.stats[k - 1, 4].item()
                if approx_kl > a.target_kl:
                    break
        if graphed:
            self.flat.step += E * nmb
            if hasattr(self.agent, "params_updated"):
                self.agent.params_updated()      # no python ran inside the replays: the packed operand copies are stale
        self.stats_h[:k].copy_(self.stats[:k], non_blocking=True)
        t_sy = time.perf_counter()
        self.host_seconds["update_enqueue"] += t_sy - t_up
        _sync()
        self.host_seconds["update_wait"] += time.perf_counter() - t_sy
        self.d2h_bytes += k * 64
        s = self.stats_h[:k].numpy()
        out = {name: float(s[k - 1, i]) for i, name in enumerate(STAT_NAMES)}
        out["clipfrac_mean"] = float(np.mean(s[:, 5].astype(np.float64)))   # np.mean(clipfracs), ppo.py:306
        out["num_updates"] = k
        out["per_update"] = s.copy()
        return out

    def _epoch_work(self, epoch, lr, k, dyn):
        B, M, nmb = self.B, self.M, self.num_minibatches
        if self.s2d and self.sort_minibatch:
            # same minibatch SETS as the reference's shuffle; rows visited in ascending address order so the frames gathered
            # by conv1 share DRAM pages / TLB entries (the sums over a minibatch are order-independent up to fp rounding)
            self.b_inds[epoch].copy_(torch.sort(self.b_inds[epoch].view(nmb, M), dim=1).values.view(B))
        for start in range(0, B, M):
            self.minibatch_update(self.b_inds[epoch, start:start + M], lr, k, dyn=self.hyper[k] if dyn else None)
            k += 1
        return k

    def _capture_epoch(self, epoch):
        from . import _lib
        if epoch == 0 and hasattr(self.agent, "params_updated"):
            self.agent.params_updated()     # the graph of epoch 0 always starts by packing the weights it was given
        l0 = _lib.load().b200rl_launch_count()
        g = torch.cuda.CUDAGraph()
        if self._graph_pool is None:
            self._graph_pool = torch.cuda.graph_pool_handle()
        with torch.cuda.graph(g, pool=self._graph_pool):
            self._epoch_work(epoch, None, epoch * self.num_minibatches, True)
        self._upd_graphs[epoch] = g
        self._upd_kernels[epoch] = _lib.load().b200rl_launch_count() - l0
        if hasattr(self.agent, "pin_workspaces"):
            self.agent.pin_workspaces()
        return g

    @torch.no_grad()
    def minibatch_update(self, mb_inds, lr, k=0, dyn=None):
        """ONE fused update on the rollout rows ``mb_inds`` (device int64): forward with the row gather folded in,
        loss + its gradient, hand-written backward, DP gradient exchange, clip + Adam (ppo.py:250-290,
        ppo_atari_multigpu.py:360-377).  ``stats[k]`` receives the logged scalars."""
        a, agent, flat, B = self.args, self.agent, self.flat, self.B
        b_obs = self.obs.view((B,) + tuple(self.obs.shape[2:]))
        b = {"actions": self.actions.view((B,) + tuple(self.actions.shape[2:])), "logprobs": self.logprobs.view(B),
             "advantages": self.advantages.view(B), "returns": self.returns.view(B), "values": self.values.view(B)}
        if not hasattr(self, "_scratch"):
            self._scratch = {}
        if self.u8_rollout:
            policy_out, value = agent.forward_train(b_obs, mb_inds, aux=self.obs_t.view(B, 64, 448))
        else:
            policy_out, value = agent.forward_train(b_obs, mb_inds)
        agent.loss_backward(policy_out, value, mb_inds, b, a, self.stats[k], self._scratch)
        if self.world_size > 1:
            self._exchange_gradients()
        if dyn is not None:      # captured: the (step, lr) scalars of update k come from the device table
            ops.clip_adam_dyn(flat.flat, flat.grad, flat.exp_avg, flat.exp_avg_sq, dyn, eps=1e-5, max_norm=a.max_grad_norm,
                              world_size=self.world_size, norm_out=self.grad_norm)
        else:
            flat.step += 1
            ops.clip_adam(flat.flat, flat.grad, flat.exp_avg, flat.exp_avg_sq, flat.step, lr,
                          eps=1e-5, max_norm=a.max_grad_norm, world_size=self.world_size,
                          norm_out=self.grad_norm)
        if hasattr(agent, "params_updated"):
            agent.params_updated()

    def _exchange_gradients(self):
        """The ONE data-parallel exchange per update: SUM of the flat gradient over ranks (the mean's 1/world_size is
        folded into clip+Adam).  Reference: cat + all_reduce + 12 copy-backs after the whole backward
        (ppo_atari_multigpu.py:360-374).  Here the fc + head gradients -- 95 % of the vector, finished first by the
        hand-written backward -- start their all-reduce on a side stream as soon as the kernel that completes them has
        run, underneath the ~2 ms of convolution backward; only the 78 k conv gradients are exchanged after the
        backward.  Both parts are elementwise sums of disjoint slices: same result as one all-reduce."""
        flat = self.flat
        tail = self.agent.grad_tail() if (self.overlap_exchange and hasattr(self.agent, "grad_tail")) else None
        if tail is None:
            self.all_reduce(flat.grad)
            return
        off, ev = tail
        main = torch.cuda.current_stream()
        if self._xchg_stream is None:
            self._xchg_stream = torch.cuda.Stream(device=self.device)
            self._xchg_done = torch.cuda.Event()
            self._bwd_done = torch.cuda.Event()
        side = self._xchg_stream
        side.wait_event(ev)                               # recorded inside backward, after the fc gradients
        with torch.cuda.stream(side):
            self.all_reduce(flat.grad[off:])
        self._bwd_done.record(main)
        side.wait_event(self._bwd_done)
        with torch.cuda.stream(side):
            self.all_reduce(flat.grad[:off])
            self._xchg_done.record(side)
        main.wait_event(self._xchg_done)

    def explained_variance(self):
        """ppo.py:295-297 on host numpy."""
        y_pred = self.values.view(-1).cpu().numpy()
        y_true = self.returns.view(-1).cpu().numpy()
        self.d2h_bytes += 2 * self.B * 4
        var_y = np.var(y_true)
        return np.nan if var_y == 0 else 1 - np.var(y_true - y_pred) / var_y
