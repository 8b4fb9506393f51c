"""CPU tests of the one-call rollout step entry point (b200rl_naturecnn_bf16_rollout_step): bad arguments are rejected
before any CUDA call, an empty batch is a no-op, and the python wrapper refuses CPU tensors (no fallback)."""
import pytest


def test_rollout_step_validates_arguments_without_gpu(lib):
    f = lib.b200rl_naturecnn_bf16_rollout_step
    ok = dict(frames=None, rm=16, cm=None, n=4, A=4, params=16, packed=16, acts=16, noise=16, action=16, logprob=16, value=16)

    def call(**kw):
        a = dict(ok, **kw)
        return f(a["frames"], a["rm"], a["cm"], a["n"], a["A"], a["params"], a["packed"], a["acts"], a["noise"], a["action"],
                 a["logprob"], a["value"], None)

    assert call(n=-1) == -1 and b"negative" in lib.b200rl_last_error()
    assert call(n=0, rm=None, params=None) == 0                      # empty batch: no-op
    for k in ("rm", "params", "packed", "acts", "noise", "action", "logprob", "value"):
        assert call(**{k: None}) == -1 and b"null" in lib.b200rl_last_error(), k
    assert call(frames=16, cm=None) == -1 and b"channel-major" in lib.b200rl_last_error()
    assert call(A=0) == -1 and call(A=24) == -1
    assert call(rm=24) == -1 and b"misaligned" in lib.b200rl_last_error()
    assert call(frames=8, cm=16) == -1 and b"misaligned" in lib.b200rl_last_error()
    assert call(n=(1 << 22) + 1) == -1 and b"too large" in lib.b200rl_last_error()


def test_rollout_step_wrapper_refuses_cpu_tensors(lib):
    import torch
    from cleanrl_b200 import ops
    tc = ops.NatureCNNBf16.__new__(ops.NatureCNNBf16)
    tc.A, tc.device = 4, torch.device("cpu")
    n = 2
    with pytest.raises(Exception):
        tc.rollout_step(None, torch.zeros(n, 441, 64, dtype=torch.uint8), None, torch.zeros(16), torch.zeros(n, 4),
                        torch.zeros(n, dtype=torch.int64), torch.zeros(n), torch.zeros(n))
