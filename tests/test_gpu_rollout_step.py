"""One-call rollout step of the bf16 NatureCNN (b200rl_naturecnn_bf16_rollout_step: conv tower with act1 / act2 in shared
memory, fc, heads + sampler) against the launch chain it replaces (frames_to_s2d_u8 + forward + categorical_sample): action,
log-probability and value bit for bit, both producer variants (raw frames / stored slot), both slot orientations written by
the raw-frame variant, and the engine's rollout buffers through rollout_resident and the grouped delta-upload collect."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _params(A, seed, dev):
    """Random NatureCNN parameters in libb200rl order, scaled per layer (1/sqrt(fan_in)) with zero-mean biases, so that
    the ReLUs zero a good fraction of the units of every layer."""
    g = torch.Generator().manual_seed(seed)
    segs = [(32 * 256, 256), (32, 0), (64 * 512, 512), (64, 0), (64 * 576, 576), (64, 0), (512 * 3136, 3136), (512, 0),
            ((A + 1) * 512, 512), (A + 1, 0)]
    out = []
    for n, fan in segs:
        t = torch.randn(n, generator=g)
        out.append(t * (1.0 / fan ** 0.5) if fan else t * 0.1)
    return torch.cat(out).to(dev)


def _chain(tc, frames, params, noise, A):
    from cleanrl_b200 import ops
    rm, cm = ops.frames_to_s2d_u8(frames)
    head = tc.forward(rm, None, params)
    a, lp, _, v = ops.categorical_sample(head[:, :A], noise, head[:, A])
    return rm, cm, a, lp, v


@pytest.mark.parametrize("A", [4, 6, 18])
def test_rollout_step_equals_chain(lib, A):
    from cleanrl_b200 import ops
    dev = torch.device("cuda")
    tc = ops.NatureCNNBf16(A, dev)
    params = _params(A, 7 + A, dev)
    tc.pack(params)
    g = torch.Generator(device=dev).manual_seed(A)
    for n in (1, 3, 127, 128, 160, 512, 1000, 1024):
        frames = torch.randint(0, 256, (n, 4, 84, 84), dtype=torch.uint8, device=dev, generator=g)
        noise = torch.empty(n, A, device=dev).exponential_(1, generator=g)
        rm, cm, a0, lp0, v0 = _chain(tc, frames, params, noise, A)
        for raw in (True, False):
            rm2 = ops.alloc_u8_rollout_rows((n, 441, 64), dev)
            cm2 = torch.full((n, 64, 448), 0xAB, dtype=torch.uint8, device=dev)
            if not raw:
                rm2.copy_(rm)
            a1 = torch.full((n,), -1, dtype=torch.int64, device=dev)
            lp1 = torch.full((n,), float("nan"), device=dev)
            v1 = torch.full((n,), float("nan"), device=dev)
            tc.rollout_step(frames if raw else None, rm2, cm2 if raw else None, params, noise, a1, lp1, v1)
            torch.cuda.synchronize()
            assert torch.equal(a1, a0), (n, raw)
            assert torch.equal(lp1, lp0), (n, raw)
            assert torch.equal(v1, v0), (n, raw)
            if raw:
                assert torch.equal(rm2, rm), n
                assert torch.equal(cm2, cm), n
        assert len(set(a0.tolist())) > 1 or n < 8


def test_rollout_step_relu_coverage(lib):
    """The random weights of the equality test leave a real fraction of every layer's units at zero (so the equality covers
    the ReLU clamp), checked on the chain's act1, act3 and hidden activations."""
    from cleanrl_b200 import ops
    dev = torch.device("cuda")
    A, n = 6, 256
    tc = ops.NatureCNNBf16(A, dev)
    params = _params(A, 13, dev)
    tc.pack(params)
    frames = torch.randint(0, 256, (n, 4, 84, 84), dtype=torch.uint8, device=dev)
    rm, _ = ops.frames_to_s2d_u8(frames)
    tc.forward(rm, None, params)
    ws = tc.acts(n, 2).view(torch.bfloat16)
    act1 = ws[:n * 12800]
    act3 = ws[n * (12800 + 5184):n * (12800 + 5184 + 3136)]
    hid = ws[n * (12800 + 5184 + 3136):n * (12800 + 5184 + 3136 + 512)]
    for t in (act1, act3, hid):
        z = float((t == 0).float().mean())
        assert 0.1 < z < 0.9, z


def _engine(N, T, fused, seed=3):
    from bench import ppo_args
    from cleanrl_b200.agents import NatureCNNAgent
    from cleanrl_b200.ppo_engine import PPOEngine
    from cleanrl_b200.synthetic_envs import SyntheticAtariVec
    dev = torch.device("cuda")
    torch.manual_seed(seed)
    spaces = SyntheticAtariVec(2, seed=1)
    spaces.single_observation_space, spaces.single_action_space = spaces.observation_space, spaces.action_space
    agent = NatureCNNAgent(spaces).to(dev)
    agent.precision = "bf16"
    eng = PPOEngine(agent, ppo_args(N, T, 4, "bf16"), (4, 84, 84), np.uint8, N, dev, gae_mode=1)
    if not fused:
        eng._fused_rollout = lambda: False
    assert eng.u8_rollout
    return eng


_KEYS = ("obs", "obs_t", "actions", "logprobs", "values")


def test_rollout_resident_equals_chain(lib):
    N, T = 512, 6
    dev = torch.device("cuda")
    pool = torch.randint(0, 256, (4, N, 4, 84, 84), dtype=torch.uint8, device=dev,
                         generator=torch.Generator(device=dev).manual_seed(5))
    outs = []
    for fused in (False, True):
        eng = _engine(N, T, fused)
        torch.manual_seed(21)
        for _ in range(2):                                  # eager warm-up + capture, then a replay
            eng.rollout_resident(pool)
        torch.cuda.synchronize()
        outs.append({k: getattr(eng, k).clone() for k in _KEYS})
    for k in _KEYS:
        assert torch.equal(outs[0][k], outs[1][k]), k


def test_grouped_delta_collect_equals_chain(lib):
    import os
    from cleanrl_b200.synthetic_envs import SyntheticAtariVec
    N, T = 256, 5
    old = os.environ.get("CLEANRL_B200_DELTA_UPLOAD")
    os.environ["CLEANRL_B200_DELTA_UPLOAD"] = "1"
    try:
        outs = []
        for fused in (False, True):
            eng = _engine(N, T, fused)
            assert eng.delta_upload
            torch.manual_seed(11)
            parts = [SyntheticAtariVec(N // 2, seed=5 + p, mode="stack", pool=8, p_done=0.05) for p in range(2)]
            obs_p = [e.reset() for e in parts]
            done_p = [np.zeros(N // 2, dtype=np.float32) for _ in parts]
            res = []
            for _ in range(2):
                obs_p, done_p = eng.collect(parts, obs_p, done_p)
                eng.finish_rollout_parts(obs_p, done_p)
                torch.cuda.synchronize()
                res.append({k: getattr(eng, k).clone() for k in _KEYS + ("next_value",)})
            outs.append(res)
    finally:
        if old is None:
            os.environ.pop("CLEANRL_B200_DELTA_UPLOAD", None)
        else:
            os.environ["CLEANRL_B200_DELTA_UPLOAD"] = old
    for it in range(2):
        for k in outs[0][it]:
            assert torch.equal(outs[0][it][k], outs[1][it][k]), (it, k)
