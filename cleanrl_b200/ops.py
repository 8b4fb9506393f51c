"""Thin torch-tensor front end over the C-ABI (device pointers + current stream).

PyTorch is plumbing here: it owns device memory and the stream; every function
below only validates arguments and enqueues libb200rl kernels on
``torch.cuda.current_stream()``.  CPU tensors are rejected loudly -- there is
no fallback path.
"""
from __future__ import annotations

import torch

from . import _lib

STAT_NAMES = ("pg_loss", "v_loss", "entropy", "old_approx_kl", "approx_kl", "clipfrac", "loss",
              "adv_mean", "adv_std")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t, dtype=None, name="tensor", allow_none=False):
    if t is None:
        if allow_none:
            return None
        raise ValueError(f"{name} is None")
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{name}: libb200rl kernels need a CUDA tensor (got {type(t).__name__} on "
                           f"{getattr(t, 'device', '?')}); there is no CPU fallback")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    return t.data_ptr()


def _contig(t, name):
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


class Workspace:
    """Grow-only device scratch buffer owned by the caller side (never by the kernels)."""

    def __init__(self, device):
        self.device = device
        self.buf = None

    def get(self, nbytes):
        if self.buf is None or self.buf.numel() < nbytes:
            self.buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=self.device)
        return self.buf


_ws = {}


def _workspace(device, key, nbytes):
    w = _ws.setdefault((device, key), Workspace(device))
    return w.get(nbytes)


def gae(rewards, values, dones, next_value, next_done, gamma, gae_lambda, mode=0, out=None):
    """advantages, returns = GAE(...)  (reference loop: cleanrl/ppo.py:218-231)."""
    lib = _lib.load()
    T, N = rewards.shape
    for n, t in (("rewards", rewards), ("values", values), ("dones", dones)):
        _contig(t, n)
        assert t.shape == (T, N), f"{n} shape {tuple(t.shape)} != {(T, N)}"
    next_value = _contig(next_value.reshape(-1), "next_value")
    next_done = _contig(next_done.reshape(-1), "next_done")
    assert next_value.numel() == N and next_done.numel() == N
    if out is None:
        adv = torch.empty_like(rewards)
        ret = torch.empty_like(rewards)
    else:
        adv, ret = out
    f = torch.float32
    rc = lib.b200rl_gae_f32(_ptr(rewards, f, "rewards"), _ptr(values, f, "values"), _ptr(dones, f, "dones"),
                            _ptr(next_value, f, "next_value"), _ptr(next_done, f, "next_done"),
                            _ptr(adv, f, "advantages"), _ptr(ret, f, "returns"),
                            T, N, float(gamma), float(gae_lambda), int(mode), _stream())
    _lib.check(rc, "gae")
    return adv, ret


def categorical_sample(logits, noise, value_in=None, out=None):
    """action, logprob, entropy[, value] from raw logits and Exp(1) noise
    (reference: Categorical(logits).sample()/log_prob/entropy, ppo_atari_envpool.py:143-149)."""
    lib = _lib.load()
    n, A = logits.shape
    assert logits.stride(1) == 1
    _contig(noise, "noise")
    assert noise.shape == (n, A)
    dev = logits.device
    if out is None:
        action = torch.empty(n, dtype=torch.int64, device=dev)
        logprob = torch.empty(n, dtype=torch.float32, device=dev)
        entropy = torch.empty(n, dtype=torch.float32, device=dev)
        value = torch.empty(n, dtype=torch.float32, device=dev) if value_in is not None else None
    else:
        action, logprob, entropy, value = out
    f = torch.float32
    ldv = 0
    if value_in is not None:
        value_in = value_in.reshape(n, -1)
        ldv = value_in.stride(0)
    rc = lib.b200rl_categorical_sample_f32(
        _ptr(logits, f, "logits"), logits.stride(0), _ptr(noise, f, "noise"),
        _ptr(value_in, f, "value_in", True), ldv, n, A,
        _ptr(action, torch.int64, "action"), _ptr(logprob, f, "logprob"),
        _ptr(entropy, f, "entropy", True), _ptr(value, f, "value_out", True), _stream())
    _lib.check(rc, "categorical_sample")
    return action, logprob, entropy, value


def categorical_eval(logits, action):
    """logprob, entropy of given actions (reference: probs.log_prob(action), probs.entropy())."""
    lib = _lib.load()
    n, A = logits.shape
    assert logits.stride(1) == 1
    action = _contig(action.reshape(-1), "action")
    if action.dtype != torch.int64:
        action = action.long()
    f = torch.float32
    logprob = torch.empty(n, dtype=f, device=logits.device)
    entropy = torch.empty(n, dtype=f, device=logits.device)
    rc = lib.b200rl_categorical_eval_f32(_ptr(logits, f, "logits"), logits.stride(0), _ptr(action, torch.int64, "action"),
                                         n, A, _ptr(logprob, f, "logprob"), _ptr(entropy, f, "entropy"), _stream())
    _lib.check(rc, "categorical_eval")
    return logprob, entropy


def ppo_loss(new_logits, new_value, mb_inds, b_actions, b_logprobs, b_advantages, b_returns, b_values,
             clip_coef, ent_coef, vf_coef, norm_adv=True, clip_vloss=True, dlogits=None, dvalue=None, stats=None):
    """Fused PPO minibatch loss + gradients (reference: cleanrl/ppo.py:250-285).
    Returns (stats f32[16] device tensor, dlogits [M,A], dvalue [M])."""
    lib = _lib.load()
    M, A = new_logits.shape
    dev = new_logits.device
    assert new_logits.stride(1) == 1
    new_value = new_value.reshape(M, -1)
    f = torch.float32
    if dlogits is None:
        dlogits = torch.empty(M, A, dtype=f, device=dev)
    if dvalue is None:
        dvalue = torch.empty(M, dtype=f, device=dev)
    dv2 = dvalue.reshape(M, -1)
    if stats is None:
        stats = torch.zeros(16, dtype=f, device=dev)
    nbytes = lib.b200rl_ppo_loss_workspace_bytes(M)
    ws = _workspace(dev, "loss", nbytes)
    if mb_inds is not None:
        _contig(mb_inds, "mb_inds")
        assert mb_inds.numel() == M
    for n_, t in (("b_actions", b_actions), ("b_logprobs", b_logprobs), ("b_advantages", b_advantages),
                  ("b_returns", b_returns), ("b_values", b_values)):
        _contig(t, n_)
    rc = lib.b200rl_ppo_loss_f32(
        _ptr(new_logits, f, "new_logits"), new_logits.stride(0), _ptr(new_value, f, "new_value"), new_value.stride(0),
        _ptr(mb_inds, torch.int64, "mb_inds", True),
        _ptr(b_actions, torch.int64, "b_actions"), _ptr(b_logprobs, f, "b_logprobs"),
        _ptr(b_advantages, f, "b_advantages"), _ptr(b_returns, f, "b_returns"), _ptr(b_values, f, "b_values"),
        M, A, float(clip_coef), float(ent_coef), float(vf_coef), int(bool(norm_adv)), int(bool(clip_vloss)),
        _ptr(dlogits, f, "dlogits"), dlogits.stride(0), _ptr(dv2, f, "dvalue"), dv2.stride(0),
        _ptr(stats, f, "stats"), ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "ppo_loss")
    return stats, dlogits, dvalue


def clip_adam(params, grads, exp_avg, exp_avg_sq, step, lr, beta1=0.9, beta2=0.999, eps=1e-5,
              max_norm=0.5, world_size=1, norm_out=None):
    """In-place fused clip_grad_norm_ + Adam step on flat f32 vectors
    (reference: cleanrl/ppo.py:289-290; DP averaging ppo_atari_multigpu.py:369-373)."""
    lib = _lib.load()
    P = params.numel()
    f = torch.float32
    for n_, t in (("params", params), ("grads", grads), ("exp_avg", exp_avg), ("exp_avg_sq", exp_avg_sq)):
        _contig(t, n_)
        assert t.numel() == P
    nbytes = lib.b200rl_clip_adam_workspace_bytes(P)
    ws = _workspace(params.device, "adam", nbytes)
    rc = lib.b200rl_clip_adam_f32(
        _ptr(params, f, "params"), _ptr(grads, f, "grads"), _ptr(exp_avg, f, "exp_avg"),
        _ptr(exp_avg_sq, f, "exp_avg_sq"), P, int(step), float(lr), float(beta1), float(beta2), float(eps),
        -1.0 if max_norm is None else float(max_norm), int(world_size),
        _ptr(norm_out, f, "norm_out", True), ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "clip_adam")
    return params


def numpy_global_shuffle(arr):
    """``np.random.shuffle(arr)`` for a contiguous int64 vector, bit-exact (same permutation, same generator state afterwards)
    but 4-6x faster: libb200rl walks numpy's own algorithm over the global RandomState's MT19937 words.  Falls back to
    numpy itself for anything else (other dtypes / strides, a replaced bit generator)."""
    import ctypes
    import numpy as np
    if not (isinstance(arr, np.ndarray) and arr.dtype == np.int64 and arr.ndim == 1 and arr.flags.c_contiguous):
        return np.random.shuffle(arr)
    st = np.random.get_state(legacy=True)
    if st[0] != "MT19937":
        return np.random.shuffle(arr)
    key = np.ascontiguousarray(st[1], dtype=np.uint32).copy()
    pos = ctypes.c_int32(int(st[2]))
    rc = _lib.load().b200rl_mt19937_shuffle_i64(key.ctypes.data, ctypes.addressof(pos), arr.ctypes.data, arr.shape[0])
    _lib.check(rc, "mt19937_shuffle")
    np.random.set_state(("MT19937", key, int(pos.value), st[3], st[4]))


def adam_step_scalars(step, lr, beta1=0.9, beta2=0.999):
    """(sqrt(1 - beta2^step), -lr / (1 - beta1^step)) as float32, computed by the library in double as ``clip_adam`` does."""
    import ctypes
    out = (ctypes.c_float * 2)()
    _lib.check(_lib.load().b200rl_adam_step_scalars(int(step), float(lr), float(beta1), float(beta2), out), "adam_step_scalars")
    return float(out[0]), float(out[1])


def clip_adam_dyn(params, grads, exp_avg, exp_avg_sq, step_scalars, beta1=0.9, beta2=0.999, eps=1e-5, max_norm=0.5,
                  world_size=1, norm_out=None):
    """``clip_adam`` with the (step, lr)-dependent scalars in device memory (``step_scalars`` f32[2], see
    ``adam_step_scalars``): what a captured CUDA graph of the update replays."""
    lib = _lib.load()
    P = params.numel()
    f = torch.float32
    for n_, t in (("params", params), ("grads", grads), ("exp_avg", exp_avg), ("exp_avg_sq", exp_avg_sq)):
        _contig(t, n_)
        assert t.numel() == P
    assert step_scalars.numel() == 2 and step_scalars.is_contiguous()
    ws = _workspace(params.device, "adam", lib.b200rl_clip_adam_workspace_bytes(P))
    rc = lib.b200rl_clip_adam_dyn_f32(
        _ptr(params, f, "params"), _ptr(grads, f, "grads"), _ptr(exp_avg, f, "exp_avg"), _ptr(exp_avg_sq, f, "exp_avg_sq"), P,
        _ptr(step_scalars, f, "step_scalars"), float(beta1), float(beta2), float(eps),
        -1.0 if max_norm is None else float(max_norm), int(world_size), _ptr(norm_out, f, "norm_out", True),
        ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "clip_adam_dyn")
    return params


# ----------------------------------------------------------------- fp32 layers
ACT = {None: 0, "none": 0, "relu": 1, "tanh": 2}


def _xdtype(x):
    if x.dtype == torch.uint8:
        return 1
    if x.dtype == torch.float32:
        return 0
    raise TypeError(f"unsupported input dtype {x.dtype} (need uint8 or float32)")


def conv2d_fwd(x, w, b, stride, act, rows=None, in_div=1.0, out=None, pad=0):
    """y = act(conv2d(x / in_div, w, padding=pad) + b), NCHW (reference: nn.Conv2d + ReLU, ppo_atari_envpool.py:126-132;
    padded 3x3: ppo_procgen.py:92-93).  ``rows`` (int64) gathers the batch dimension of x without materialising it (ppo.py:250)."""
    lib = _lib.load()
    _contig(x, "x"); _contig(w, "w")
    Cout, Cin, KH, KW = w.shape
    H, W = x.shape[-2:]
    assert x.shape[-3] == Cin
    n = rows.numel() if rows is not None else x.shape[0]
    OH, OW = (H + 2 * pad - KH) // stride + 1, (W + 2 * pad - KW) // stride + 1
    if out is None:
        out = torch.empty(n, Cout, OH, OW, dtype=torch.float32, device=x.device)
    rc = lib.b200rl_conv2d_fwd_pad_f32(_ptr(x, None, "x"), _xdtype(x), _ptr(rows, torch.int64, "rows", True), float(in_div),
                                       _ptr(w, torch.float32, "w"), _ptr(b, torch.float32, "b", True),
                                       _ptr(out, torch.float32, "y"), n, Cin, H, W, Cout, KH, KW, stride, int(pad), ACT[act], _stream())
    _lib.check(rc, "conv2d_fwd")
    return out


def conv2d_bwd_data(dy, w, x_post, prev_act, stride, out=None, pad=0, in_hw=None):
    """dx of the convolution; ``x_post`` / ``prev_act`` fold the derivative of the activation that produced the layer
    input (``prev_act=None``: pass ``in_hw=(H, W)`` instead of ``x_post``)."""
    lib = _lib.load()
    _contig(dy, "dy"); _contig(w, "w")
    Cout, Cin, KH, KW = w.shape
    n = dy.shape[0]
    H, W = x_post.shape[-2:] if x_post is not None else in_hw
    if out is None:
        out = torch.empty(n, Cin, H, W, dtype=torch.float32, device=dy.device)
    rc = lib.b200rl_conv2d_bwd_data_pad_f32(_ptr(dy, torch.float32, "dy"), _ptr(w, torch.float32, "w"),
                                            _ptr(x_post, torch.float32, "x_post", True), ACT[prev_act] if x_post is not None else 0,
                                            _ptr(out, torch.float32, "dx"), n, Cin, H, W, Cout, KH, KW, stride, int(pad), _stream())
    _lib.check(rc, "conv2d_bwd_data")
    return out


def conv2d_bwd_weight(x, dy, dw, db, stride, rows=None, in_div=1.0, pad=0):
    lib = _lib.load()
    _contig(x, "x"); _contig(dy, "dy"); _contig(dw, "dw")
    Cout, Cin, KH, KW = dw.shape
    H, W = x.shape[-2:]
    n = dy.shape[0]
    nbytes = lib.b200rl_conv2d_bwd_weight_pad_workspace_bytes(n, Cin, H, W, Cout, KH, KW, stride, int(pad))
    ws = _workspace(x.device, "wgrad", nbytes)
    rc = lib.b200rl_conv2d_bwd_weight_pad_f32(_ptr(x, None, "x"), _xdtype(x), _ptr(rows, torch.int64, "rows", True),
                                              float(in_div), _ptr(dy, torch.float32, "dy"), _ptr(dw, torch.float32, "dw"),
                                              _ptr(db, torch.float32, "db", True), n, Cin, H, W, Cout, KH, KW, stride, int(pad),
                                              ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "conv2d_bwd_weight")


def linear_fwd(x, w, b, act, rows=None, out=None):
    """y = act(x @ w.T + b) (reference: nn.Linear + activation)."""
    lib = _lib.load()
    _contig(x, "x"); _contig(w, "w")
    out_f, in_f = w.shape
    x2 = x.reshape(x.shape[0], -1)
    assert x2.shape[1] == in_f, f"linear_fwd: x has {x2.shape[1]} features, w expects {in_f}"
    n = rows.numel() if rows is not None else x2.shape[0]
    if out is None:
        out = torch.empty(n, out_f, dtype=torch.float32, device=x.device)
    rc = lib.b200rl_linear_fwd_f32(_ptr(x2, torch.float32, "x"), _ptr(rows, torch.int64, "rows", True),
                                   _ptr(w, torch.float32, "w"), _ptr(b, torch.float32, "b", True),
                                   _ptr(out, torch.float32, "y"), n, in_f, out_f, ACT[act], _stream())
    _lib.check(rc, "linear_fwd")
    return out


def linear_bwd_data(dy, w, x_post, prev_act, out=None):
    lib = _lib.load()
    _contig(dy, "dy"); _contig(w, "w")
    out_f, in_f = w.shape
    n = dy.shape[0]
    if out is None:
        out = torch.empty(n, in_f, dtype=torch.float32, device=dy.device)
    rc = lib.b200rl_linear_bwd_data_f32(_ptr(dy, torch.float32, "dy"), _ptr(w, torch.float32, "w"),
                                        _ptr(x_post, torch.float32, "x_post", True), ACT[prev_act],
                                        _ptr(out, torch.float32, "dx"), n, in_f, out_f, _stream())
    _lib.check(rc, "linear_bwd_data")
    return out


def linear_bwd_weight(x, dy, dw, db, rows=None):
    lib = _lib.load()
    _contig(x, "x"); _contig(dy, "dy"); _contig(dw, "dw")
    out_f, in_f = dw.shape
    n = dy.shape[0]
    nbytes = lib.b200rl_linear_bwd_weight_workspace_bytes(n, in_f, out_f)
    ws = _workspace(x.device, "wgrad", nbytes)
    rc = lib.b200rl_linear_bwd_weight_f32(_ptr(x, torch.float32, "x"), _ptr(rows, torch.int64, "rows", True),
                                          _ptr(dy, torch.float32, "dy"), _ptr(dw, torch.float32, "dw"),
                                          _ptr(db, torch.float32, "db", True), n, in_f, out_f,
                                          ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "linear_bwd_weight")


# ------------------------------------------------------------------ IMPALA-CNN glue
def maxpool3s2_fwd(x):
    """max_pool2d(x, kernel_size=3, stride=2, padding=1) on NCHW fp32 (ppo_procgen.py:113); returns (y, argmax u8)."""
    lib = _lib.load()
    _contig(x, "x")
    n, C, H, W = x.shape
    y = torch.empty(n, C, (H + 1) // 2, (W + 1) // 2, dtype=torch.float32, device=x.device)
    arg = torch.empty(y.shape, dtype=torch.uint8, device=x.device)
    _lib.check(lib.b200rl_maxpool3s2_fwd_f32(_ptr(x, torch.float32, "x"), n * C, H, W, _ptr(y, torch.float32, "y"),
                                             _ptr(arg, torch.uint8, "argmax"), _stream()), "maxpool_fwd")
    return y, arg


def maxpool3s2_bwd(dy, arg, in_hw):
    lib = _lib.load()
    _contig(dy, "dy")
    n, C = dy.shape[:2]
    H, W = in_hw
    dx = torch.empty(n, C, H, W, dtype=torch.float32, device=dy.device)
    _lib.check(lib.b200rl_maxpool3s2_bwd_f32(_ptr(dy, torch.float32, "dy"), _ptr(arg, torch.uint8, "argmax"), n * C, H, W,
                                             _ptr(dx, torch.float32, "dx"), _stream()), "maxpool_bwd")
    return dx


def relu(x):
    lib = _lib.load()
    y = torch.empty_like(_contig(x, "x"))
    _lib.check(lib.b200rl_relu_f32(_ptr(x, torch.float32, "x"), x.numel(), _ptr(y, torch.float32, "y"), _stream()), "relu")
    return y


def relu_bwd(dy, x, extra=None):
    """dx = dy * (x > 0) [+ extra]."""
    lib = _lib.load()
    dx = torch.empty_like(_contig(dy, "dy"))
    _lib.check(lib.b200rl_relu_bwd_f32(_ptr(dy, torch.float32, "dy"), _ptr(_contig(x, "x"), torch.float32, "x"),
                                       _ptr(extra, torch.float32, "extra", True), dy.numel(), _ptr(dx, torch.float32, "dx"),
                                       _stream()), "relu_bwd")
    return dx


def add(a, b):
    lib = _lib.load()
    y = torch.empty_like(_contig(a, "a"))
    _lib.check(lib.b200rl_add_f32(_ptr(a, torch.float32, "a"), _ptr(_contig(b, "b"), torch.float32, "b"), a.numel(),
                                  _ptr(y, torch.float32, "y"), _stream()), "add")
    return y


def nhwc_to_nchw_u8(x, rows=None):
    """uint8 frames [*, H, W, C] (optionally gathered through int64 ``rows``) -> [n, C, H, W] (ppo_procgen.py:143 permute)."""
    lib = _lib.load()
    _contig(x, "x")
    H, W, C = x.shape[-3:]
    n = rows.numel() if rows is not None else x.shape[0]
    y = torch.empty(n, C, H, W, dtype=torch.uint8, device=x.device)
    _lib.check(lib.b200rl_nhwc_to_nchw_u8(_ptr(x, torch.uint8, "x"), _ptr(rows, torch.int64, "rows", True), n, H, W, C,
                                          _ptr(y, torch.uint8, "y"), _stream()), "nhwc_to_nchw")
    return y


# ------------------------------------------------------------------------ LSTM cell
def lstm_mask_state(h, c, done, out=None):
    """(h', c') = (1 - done) * (h, c): the state reset of cleanrl/ppo_atari_lstm.py:137-142, [n, H] fp32."""
    lib = _lib.load()
    n, H = h.shape
    f = torch.float32
    hm, cm = out if out is not None else (torch.empty_like(h), torch.empty_like(c))
    rc = lib.b200rl_lstm_mask_state_f32(_ptr(_contig(h, "h"), f, "h"), _ptr(_contig(c, "c"), f, "c"),
                                        _ptr(_contig(done, "done"), f, "done"), n, H, _ptr(hm, f, "hm"), _ptr(cm, f, "cm"), _stream())
    _lib.check(rc, "lstm_mask_state")
    return hm, cm


def lstm_cell_fwd(gates_x, gates_h, c_masked, h_out, c_out, save=None):
    """One LSTM step from the two gate GEMMs (gate order i, f, g, o); ``save`` [n, 5H] keeps what the backward needs."""
    lib = _lib.load()
    n, H = c_masked.shape
    f = torch.float32
    for nm, t in (("gates_x", gates_x), ("gates_h", gates_h), ("c_masked", c_masked), ("h_out", h_out), ("c_out", c_out)):
        _contig(t, nm)
    assert gates_x.shape == (n, 4 * H) and gates_h.shape == (n, 4 * H)
    rc = lib.b200rl_lstm_cell_fwd_f32(_ptr(gates_x, f, "gates_x"), _ptr(gates_h, f, "gates_h"), _ptr(c_masked, f, "c_masked"), n, H,
                                      _ptr(h_out, f, "h_out"), _ptr(c_out, f, "c_out"), _ptr(save, f, "save", True), _stream())
    _lib.check(rc, "lstm_cell_fwd")


def lstm_cell_bwd(dh_heads, dh_rec_raw, done_next, dc_rec, save, c_masked, done, dgates, dc_rec_out):
    """One step of back-propagation through time (see include/b200rl.h)."""
    lib = _lib.load()
    n, H = c_masked.shape
    f = torch.float32
    for nm, t in (("dh_heads", dh_heads), ("save", save), ("c_masked", c_masked), ("done", done), ("dgates", dgates),
                  ("dc_rec_out", dc_rec_out)):
        _contig(t, nm)
    rc = lib.b200rl_lstm_cell_bwd_f32(_ptr(dh_heads, f, "dh_heads"), _ptr(dh_rec_raw, f, "dh_rec_raw", True),
                                      _ptr(done_next, f, "done_next", True), _ptr(dc_rec, f, "dc_rec", True), _ptr(save, f, "save"),
                                      _ptr(c_masked, f, "c_masked"), _ptr(done, f, "done"), n, H, _ptr(dgates, f, "dgates"),
                                      _ptr(dc_rec_out, f, "dc_rec_out"), _stream())
    _lib.check(rc, "lstm_cell_bwd")


# ------------------------------------------------------ NatureCNN bf16 (tcgen05) plan
class NatureCNNBf16:
    """Owns the packed bf16 weights and activation workspaces of the tensor-core NatureCNN path."""

    def __init__(self, A, device):
        lib = _lib.load()
        self.A, self.device = int(A), device
        self.param_count = lib.b200rl_naturecnn_param_count(self.A)
        self.packed = torch.empty(lib.b200rl_naturecnn_bf16_packed_bytes(self.A), dtype=torch.uint8, device=device)
        self._acts = {}          # (n, fmt) -> workspace, in least-recently-used order
        self._pinned = set()     # keys referenced by captured CUDA graphs (raw pointers baked in): never evicted
        self._ws = None

    MAX_UNPINNED = 4

    def pin(self):
        """Called by the engine after a CUDA-graph capture: every workspace that exists now may be referenced by a
        graph (and by its baked CUtensorMaps) through its raw device pointer, so it must outlive the graph."""
        self._pinned.update(self._acts.keys())

    def acts(self, n, fmt):
        lib = _lib.load()
        key = (n, fmt)
        buf = self._acts.pop(key, None)
        if buf is None:
            # bounded cache of batch shapes: evict least-recently-used workspaces that no graph can reference
            unpinned = [k for k in self._acts if k not in self._pinned]
            while len(unpinned) >= self.MAX_UNPINNED:
                del self._acts[unpinned.pop(0)]
            # zero-initialised: the padded-grid gradient buffers rely on never-written positions being 0
            buf = torch.zeros(lib.b200rl_naturecnn_bf16_acts_bytes(n, fmt), dtype=torch.uint8, device=self.device)
        self._acts[key] = buf    # most recently used = last
        return buf

    @staticmethod
    def obs_format(obs):
        if obs.dtype == torch.uint8 and obs.dim() >= 4 and tuple(obs.shape[-3:]) == (4, 84, 84):
            return 0
        if obs.dtype == torch.bfloat16 and tuple(obs.shape[-3:]) == (21, 21, 64):
            return 1
        if obs.dtype == torch.uint8 and tuple(obs.shape[-2:]) == (441, 64):
            return 2
        raise TypeError("tensor-core NatureCNN path consumes uint8 [*,4,84,84] frames, uint8 space-to-depth rollout rows "
                        f"[*,441,64] or space-to-depth bf16 [*,21,21,64] (got {obs.dtype} {tuple(obs.shape)})")

    def pack(self, flat_params):
        lib = _lib.load()
        rc = lib.b200rl_naturecnn_bf16_pack(_ptr(flat_params, torch.float32, "params"), self.A,
                                            self.packed.data_ptr(), _stream())
        _lib.check(rc, "naturecnn_bf16_pack")

    def forward(self, obs, rows, flat_params, head_out=None):
        lib = _lib.load()
        fmt = self.obs_format(obs)
        _contig(obs, "obs")
        n = rows.numel() if rows is not None else obs.shape[0]
        if head_out is None:
            head_out = torch.empty(n, self.A + 1, dtype=torch.float32, device=self.device)
        rc = lib.b200rl_naturecnn_bf16_forward(_ptr(obs, None, "obs"), fmt, _ptr(rows, torch.int64, "rows", True), n, self.A,
                                               _ptr(flat_params, torch.float32, "params"), self.packed.data_ptr(),
                                               self.acts(n, fmt).data_ptr(), _ptr(head_out, torch.float32, "head_out"), _stream())
        _lib.check(rc, "naturecnn_bf16_forward")
        return head_out

    def rollout_step(self, frames, slot_rm, slot_cm, flat_params, noise, action, logprob, value):
        """One rollout policy step on the uint8 rollout layout in one native call (conv tower -> fc -> heads + sampler):
        ``frames`` uint8 [n,4,84,84] are converted into both slot orientations (``slot_rm`` [n,441,64], ``slot_cm``
        [n,64,448]) on the way; ``frames=None``: ``slot_rm`` already holds them.  Writes ``action`` (int64),
        ``logprob`` and ``value`` [n]; bit-identical to frames_to_s2d_u8 + forward + categorical_sample."""
        lib = _lib.load()
        n = slot_rm.shape[0]
        _contig(slot_rm, "slot_rm")
        if tuple(slot_rm.shape[1:]) != (441, 64) or slot_rm.dtype != torch.uint8:
            raise TypeError(f"slot_rm must be uint8 [n,441,64] (got {slot_rm.dtype} {tuple(slot_rm.shape)})")
        if frames is not None:
            _contig(frames, "frames"); _contig(slot_cm, "slot_cm")
            if tuple(frames.shape) != (n, 4, 84, 84) or tuple(slot_cm.shape) != (n, 64, 448):
                raise ValueError("frames [n,4,84,84] and slot_cm [n,64,448] must match slot_rm's n")
        _contig(noise, "noise")
        assert tuple(noise.shape) == (n, self.A)
        for nm, t in (("action", action), ("logprob", logprob), ("value", value)):
            _contig(t, nm)
            assert t.shape[0] == n, nm
        f = torch.float32
        rc = lib.b200rl_naturecnn_bf16_rollout_step(
            _ptr(frames, torch.uint8, "frames", True), _ptr(slot_rm, torch.uint8, "slot_rm"),
            _ptr(slot_cm if frames is not None else None, torch.uint8, "slot_cm", True), n, self.A,
            _ptr(flat_params, f, "params"), self.packed.data_ptr(), self.acts(n, 2).data_ptr(), _ptr(noise, f, "noise"),
            _ptr(action, torch.int64, "action"), _ptr(logprob, f, "logprob"), _ptr(value, f, "value"), _stream())
        _lib.check(rc, "naturecnn_bf16_rollout_step")

    def grad_tail_offset(self):
        """Element offset from which the flat gradient (fc + heads, 95 % of it) is final when ``tail_event`` fires."""
        return int(_lib.load().b200rl_naturecnn_grad_tail_offset(self.A))

    def backward(self, obs, rows, flat_params, dhead, flat_grads, tail_event=None, obs_aux=None):
        """``obs_aux``: the channel-major uint8 copy [*,64,448] of a uint8 space-to-depth rollout (format 2)."""
        lib = _lib.load()
        fmt = self.obs_format(obs)
        if fmt == 2:
            if obs_aux is None or obs_aux.dtype != torch.uint8 or tuple(obs_aux.shape[-2:]) != (64, 448) or \
                    obs_aux.shape[0] != obs.shape[0]:
                raise ValueError("uint8 rollout rows need their channel-major copy [*,64,448] (obs_aux) for the backward pass")
            _contig(obs_aux, "obs_aux")
        n = dhead.shape[0]
        _contig(dhead, "dhead")
        nbytes = lib.b200rl_naturecnn_bf16_workspace_bytes(n, self.A)
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        rc = lib.b200rl_naturecnn_bf16_backward(_ptr(obs, None, "obs"), _ptr(obs_aux, None, "obs_aux", True), fmt,
                                                _ptr(rows, torch.int64, "rows", True), n, self.A,
                                                _ptr(flat_params, torch.float32, "params"), self.packed.data_ptr(),
                                                self.acts(n, fmt).data_ptr(), _ptr(dhead, torch.float32, "dhead"),
                                                _ptr(flat_grads, torch.float32, "grads"),
                                                self._ws.data_ptr(), self._ws.numel(),
                                                tail_event.cuda_event if tail_event is not None else None, _stream())
        _lib.check(rc, "naturecnn_bf16_backward")


def frames_to_s2d(obs_u8, out=None, rows=None):
    """uint8 [n,4,84,84] frames -> bf16 [n,21,21,64] space-to-depth frames (once per env step)."""
    lib = _lib.load()
    _contig(obs_u8, "obs")
    n = rows.numel() if rows is not None else obs_u8.shape[0]
    if out is None:
        out = torch.empty(n, 21, 21, 64, dtype=torch.bfloat16, device=obs_u8.device)
    rc = lib.b200rl_frames_to_s2d_bf16(_ptr(obs_u8, torch.uint8, "obs"), _ptr(rows, torch.int64, "rows", True), n,
                                       _ptr(out, torch.bfloat16, "out"), _stream())
    _lib.check(rc, "frames_to_s2d")
    return out


def alloc_u8_rollout_rows(shape, device):
    """uint8 row-major rollout rows [..., 441, 64] with 256 bytes of slack behind the last frame: conv1 reads a frame as
    221 rows of 128 bytes (pairs of grid positions), and the second half of the last pair row lies 64 bytes past the frame."""
    n = 1
    for d in shape:
        n *= int(d)
    flat = torch.zeros(n + 256, dtype=torch.uint8, device=device)
    return flat[:n].view(*shape)


def frames_to_s2d_u8(obs_u8, out_rm=None, out_cm=None, rows=None):
    """uint8 [n,4,84,84] frames -> uint8 space-to-depth rollout rows: row-major [n,441,64] (conv1 forward on the integer
    tensor cores) and channel-major [n,64,448] (conv1 weight gradient); once per env step, 1 byte per pixel each."""
    lib = _lib.load()
    _contig(obs_u8, "obs")
    n = rows.numel() if rows is not None else obs_u8.shape[0]
    if out_rm is None:
        out_rm = alloc_u8_rollout_rows((n, 441, 64), obs_u8.device)
    if out_cm is None:
        out_cm = torch.empty(n, 64, 448, dtype=torch.uint8, device=obs_u8.device)
    _contig(out_rm, "out_rm"); _contig(out_cm, "out_cm")
    assert out_rm.shape[0] == n and out_cm.shape[0] == n
    rc = lib.b200rl_frames_to_s2d_u8(_ptr(obs_u8, torch.uint8, "obs"), _ptr(rows, torch.int64, "rows", True), n,
                                     _ptr(out_rm, torch.uint8, "out_rm"), _ptr(out_cm, torch.uint8, "out_cm"), _stream())
    _lib.check(rc, "frames_to_s2d_u8")
    return out_rm, out_cm


def frames_delta_s2d_u8(new_planes, prev_rm, prev_cm, out_rm, out_cm, full_slot=None, full_frames=None):
    """Rollout slot t from slot t-1 and the newest frame plane of every env (frame-stack delta upload, csrc/frame_stack.cu):
    ``new_planes`` u8 [n,7056]; envs with ``full_slot[i] = k >= 0`` take all four planes from ``full_frames[k]`` instead."""
    lib = _lib.load()
    n = new_planes.shape[0]
    for nm, t in (("new_planes", new_planes), ("prev_rm", prev_rm), ("prev_cm", prev_cm), ("out_rm", out_rm), ("out_cm", out_cm)):
        _contig(t, nm)
        assert t.shape[0] == n, nm
    if full_slot is not None:
        _contig(full_slot, "full_slot"); _contig(full_frames, "full_frames")
        assert full_slot.shape[0] == n
    rc = lib.b200rl_frames_delta_s2d_u8(_ptr(new_planes, torch.uint8, "new_planes"), _ptr(full_slot, torch.int32, "full_slot", True),
                                        _ptr(full_frames, torch.uint8, "full_frames", True), _ptr(prev_rm, torch.uint8, "prev_rm"),
                                        _ptr(prev_cm, torch.uint8, "prev_cm"), n, _ptr(out_rm, torch.uint8, "out_rm"),
                                        _ptr(out_cm, torch.uint8, "out_cm"), _stream())
    _lib.check(rc, "frames_delta_s2d_u8")


def h2d_rows_async(dst, src_ptr, src_pitch, row_bytes, rows, stream=None):
    """``rows`` rows of ``row_bytes`` from pitched host memory at address ``src_ptr`` into the dense device tensor ``dst``."""
    lib = _lib.load()
    assert dst.is_contiguous() and dst.numel() * dst.element_size() >= rows * row_bytes
    rc = lib.b200rl_h2d_rows_async(dst.data_ptr(), src_ptr, src_pitch, row_bytes, rows,
                                   stream.cuda_stream if stream is not None else _stream())
    _lib.check(rc, "h2d_rows_async")


class StackDeltaTracker:
    """Host side of the frame-stack delta upload for one vector env of ``n`` envs (b200rl_stackdelta_*): private mirror of
    every env's last observation + worker threads that verify, off the critical path, that the newest observation really
    is the previous one shifted by a plane for every env not flagged done."""

    def __init__(self, n, planes=4, plane_bytes=7056, threads=None, pinned=True):
        lib = _lib.load()
        if threads is None:
            import os
            ranks = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))        # one process per GPU shares the host cores
            threads = int(os.environ.get("CLEANRL_B200_HOST_THREADS", min(8, max(2, (os.cpu_count() or 2) // (4 * ranks)))))
        self.n, self.planes, self.plane_bytes, self.threads = int(n), int(planes), int(plane_bytes), int(threads)
        self._h = lib.b200rl_stackdelta_create(self.n, self.planes, self.plane_bytes, int(threads))
        if not self._h:
            _lib.check(-1, "stackdelta_create")
        pin = pinned and torch.cuda.is_available()
        mk = lambda shape, dt: (torch.zeros(shape, dtype=dt).pin_memory() if pin else torch.zeros(shape, dtype=dt))
        self.new_h = mk((self.n, self.plane_bytes), torch.uint8)
        self.full_h = mk((self.n, self.planes * self.plane_bytes), torch.uint8)
        self.slot_h = mk((self.n,), torch.int32)
        self.mis_h = torch.zeros(self.n, dtype=torch.int32)
        self._pending = False

    def begin(self, obs, done=None, pack_new=True):
        """obs: uint8 ndarray [n, planes, ...] whose planes are contiguous per env (any env stride).  Returns the number of
        envs staged as full frames; ``slot_h`` / ``full_h`` (and ``new_h`` when ``pack_new``) are filled on return."""
        lib = _lib.load()
        assert obs.dtype.name == "uint8" and obs.shape[0] == self.n
        itemsz = self.planes * self.plane_bytes
        inner = 1
        for d, st in zip(obs.shape[:0:-1], obs.strides[:0:-1]):
            assert st == inner, "observation planes must be contiguous per env"
            inner *= d
        assert inner == itemsz, "observation size does not match the tracker geometry"
        d32 = None
        if done is not None:
            import numpy as np
            d32 = np.ascontiguousarray(done, dtype=np.float32).reshape(-1)
            assert d32.shape[0] == self.n
        self._keep = (obs, d32)                                  # the workers read these until wait()
        k = lib.b200rl_stackdelta_begin(self._h, obs.__array_interface__["data"][0], int(obs.strides[0]),
                                        d32.__array_interface__["data"][0] if d32 is not None else None,
                                        self.new_h.data_ptr() if pack_new else None, self.full_h.data_ptr(), self.slot_h.data_ptr())
        if k < 0:
            _lib.check(int(k), "stackdelta_begin")
        self._pending = True
        return int(k)

    def wait(self):
        """Join the verification; returns the (ascending) indices of envs that were NOT a shifted stack although not done."""
        if not self._pending:
            return self.mis_h[:0].numpy()
        m = _lib.load().b200rl_stackdelta_wait(self._h, self.mis_h.data_ptr())
        self._pending = False
        self._keep = None
        if m < 0:
            _lib.check(int(m), "stackdelta_wait")
        return self.mis_h[:int(m)].numpy()

    def invalidate(self):
        if self._pending:
            self.wait()
        _lib.load().b200rl_stackdelta_invalidate(self._h)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                _lib.load().b200rl_stackdelta_destroy(h)
            except Exception:
                pass


# ----------------------------------------------------------- diagonal Gaussian policy
def gaussian_sample(mean, logstd, noise, value_in=None, out=None):
    """action, logprob, entropy[, value] for Normal(mean, exp(logstd)) with caller-supplied N(0,1) noise
    (reference: ppo_continuous_action.py:134-141)."""
    lib = _lib.load()
    n, D = mean.shape
    assert mean.stride(1) == 1
    _contig(noise, "noise"); _contig(logstd, "logstd")
    dev = mean.device
    f = torch.float32
    if out is None:
        action = torch.empty(n, D, dtype=f, device=dev)
        logprob = torch.empty(n, dtype=f, device=dev)
        entropy = torch.empty(n, dtype=f, device=dev)
        value = torch.empty(n, dtype=f, device=dev) if value_in is not None else None
    else:
        action, logprob, entropy, value = out
    ldv = 0
    if value_in is not None:
        value_in = value_in.reshape(n, -1)
        ldv = value_in.stride(0)
    rc = lib.b200rl_gaussian_sample_f32(_ptr(mean, f, "mean"), mean.stride(0), _ptr(logstd, f, "logstd"), _ptr(noise, f, "noise"),
                                        _ptr(value_in, f, "value_in", True), ldv, n, D, _ptr(action, f, "action"),
                                        _ptr(logprob, f, "logprob"), _ptr(entropy, f, "entropy", True),
                                        _ptr(value, f, "value_out", True), _stream())
    _lib.check(rc, "gaussian_sample")
    return action, logprob, entropy, value


def gaussian_eval(mean, logstd, action):
    lib = _lib.load()
    n, D = mean.shape
    f = torch.float32
    action = _contig(action.reshape(n, D), "action")
    logprob = torch.empty(n, dtype=f, device=mean.device)
    entropy = torch.empty(n, dtype=f, device=mean.device)
    rc = lib.b200rl_gaussian_eval_f32(_ptr(mean, f, "mean"), mean.stride(0), _ptr(logstd, f, "logstd"), _ptr(action, f, "action"),
                                      n, D, _ptr(logprob, f, "logprob"), _ptr(entropy, f, "entropy"), _stream())
    _lib.check(rc, "gaussian_eval")
    return logprob, entropy


def ppo_loss_gaussian(new_mean, logstd, new_value, mb_inds, b_actions, b_logprobs, b_advantages, b_returns, b_values,
                      clip_coef, ent_coef, vf_coef, norm_adv=True, clip_vloss=True, dmean=None, dlogstd=None, dvalue=None,
                      stats=None):
    """Continuous-action PPO loss + gradients (reference: ppo_continuous_action.py:262-300)."""
    lib = _lib.load()
    M, D = new_mean.shape
    dev = new_mean.device
    f = torch.float32
    new_value = new_value.reshape(M, -1)
    if dmean is None:
        dmean = torch.empty(M, D, dtype=f, device=dev)
    if dlogstd is None:
        dlogstd = torch.empty(D, dtype=f, device=dev)
    if dvalue is None:
        dvalue = torch.empty(M, dtype=f, device=dev)
    dv2 = dvalue.reshape(M, -1)
    if stats is None:
        stats = torch.zeros(16, dtype=f, device=dev)
    ws = _workspace(dev, "gloss", lib.b200rl_ppo_loss_gaussian_workspace_bytes(M))
    rc = lib.b200rl_ppo_loss_gaussian_f32(
        _ptr(new_mean, f, "new_mean"), new_mean.stride(0), _ptr(logstd, f, "logstd"),
        _ptr(new_value, f, "new_value"), new_value.stride(0), _ptr(mb_inds, torch.int64, "mb_inds", True),
        _ptr(b_actions, f, "b_actions"), _ptr(b_logprobs, f, "b_logprobs"), _ptr(b_advantages, f, "b_advantages"),
        _ptr(b_returns, f, "b_returns"), _ptr(b_values, f, "b_values"), M, D, float(clip_coef), float(ent_coef),
        float(vf_coef), int(bool(norm_adv)), int(bool(clip_vloss)), _ptr(dmean, f, "dmean"), dmean.stride(0),
        _ptr(dlogstd, f, "dlogstd"), _ptr(dv2, f, "dvalue"), dv2.stride(0), _ptr(stats, f, "stats"),
        ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "ppo_loss_gaussian")
    return stats, dmean, dlogstd, dvalue


# ------------------------------------------------------------------------ DQN
def dqn_td_loss(q, q_target_next, actions, rewards, dones, gamma, huber=False, dq=None, stats=None):
    """TD target, loss and dL/dQ (reference: dqn_atari.py:220-224).  Returns (stats[2] = td_loss, mean Q; dq)."""
    lib = _lib.load()
    B, A = q.shape
    f = torch.float32
    if dq is None:
        dq = torch.empty(B, A, dtype=f, device=q.device)
    if stats is None:
        stats = torch.zeros(2, dtype=f, device=q.device)
    ws = _workspace(q.device, "td", lib.b200rl_dqn_td_loss_workspace_bytes(B))
    rc = lib.b200rl_dqn_td_loss_f32(_ptr(q, f, "q"), q.stride(0), _ptr(q_target_next, f, "q_target_next"), q_target_next.stride(0),
                                    _ptr(_contig(actions.reshape(-1), "actions"), torch.int64, "actions"),
                                    _ptr(_contig(rewards.reshape(-1), "rewards"), f, "rewards"),
                                    _ptr(_contig(dones.reshape(-1), "dones"), f, "dones"), B, A, float(gamma), int(bool(huber)),
                                    _ptr(dq, f, "dq"), dq.stride(0), _ptr(stats, f, "stats"), ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "dqn_td_loss")
    return stats, dq


def argmax(q):
    lib = _lib.load()
    n, A = q.shape
    out = torch.empty(n, dtype=torch.int64, device=q.device)
    rc = lib.b200rl_argmax_f32(_ptr(q, torch.float32, "q"), q.stride(0), n, A, _ptr(out, torch.int64, "out"), _stream())
    _lib.check(rc, "argmax")
    return out
