"""Agent nn.Modules with the reference's surface, executed by libb200rl kernels.

Surface kept (SURVEY.md 8b): ctor ``Agent(envs)`` reading
``envs.single_observation_space`` / ``envs.single_action_space``; sub-module
names (=> identical ``state_dict`` keys); ``get_value(x)`` and
``get_action_and_value(x, action=None)`` returning
``(action i64 [n], logprob f32 [n], entropy f32 [n], value f32 [n,1])``.
Initialisation calls torch's ``orthogonal_`` in the reference's layer order so
a seed yields the reference's weights (cleanrl/ppo_atari_envpool.py:117-138,
cleanrl/ppo.py:94-116).

Forward/backward never touch autograd or cuDNN: they are explicit kernel
launches on CUDA tensors, and raise on CPU tensors (no fallback).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn

from . import nets, ops


def layer_init(layer, std=np.sqrt(2), bias_const=0.0):
    torch.nn.init.orthogonal_(layer.weight, std)
    torch.nn.init.constant_(layer.bias, bias_const)
    return layer


def _exp_noise(n, A, device):
    # what torch.multinomial consumes internally: empty_like(probs).exponential_(1)
    return torch.empty(n, A, dtype=torch.float32, device=device).exponential_(1)


_exp_noise.graph_safe = True      # device-generator draw: capturable in a CUDA graph
_exp_noise.inplace = lambda buf: buf.exponential_(1)     # same generator consumption as the out-of-place draw


class KernelAgent(nn.Module):
    """Shared plumbing: flat parameter binding + categorical head."""

    def __init__(self):
        super().__init__()
        self._flat = None
        self.noise_fn = _exp_noise   # tests may inject CPU-generator noise for cross-device parity

    # -- flat-buffer binding ------------------------------------------------
    def _param_order(self):
        return list(self.parameters())

    def bind(self):
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("cleanrl_b200 agents execute on CUDA only (libb200rl kernels); "
                               f"parameters are on {dev}. There is no CPU fallback.")
        self._flat = nets.FlatParams(self._param_order(), dev)
        self._build_plan()
        return self._flat

    @property
    def flat(self):
        p = next(self.parameters())
        if self._flat is None or self._flat.flat.device != p.device or \
                p.data_ptr() < self._flat.flat.data_ptr() or \
                p.data_ptr() >= self._flat.flat.data_ptr() + self._flat.flat.numel() * 4:
            self.bind()
        return self._flat

    # -- to be provided by subclasses --------------------------------------
    def _build_plan(self):
        raise NotImplementedError

    def _forward_heads(self, x, rows=None, keep=False):
        """returns (logits view [n,A] , value view [n] ) possibly strided"""
        raise NotImplementedError

    def backward(self, dlogits, dvalue):
        raise NotImplementedError

    # -- engine hooks (one policy step / one minibatch loss+backward) ---------------
    action_dim = 0          # 0 = discrete (int64 actions [n]); D > 0 = continuous (f32 actions [n, D])

    @property
    def graph_capturable(self):
        """May the engine capture the per-step device work (frame conversion, network, sampler) in CUDA graphs?"""
        return getattr(self, "precision", "bf16") == "bf16" or not hasattr(self, "network")

    @property
    def graph_friendly(self):
        """... and may the noise draw be captured too (device generator)?  Needed for whole-rollout graphs."""
        return getattr(self.noise_fn, "graph_safe", False) and self.graph_capturable

    def noise_shape(self, n):
        return (n, self.num_actions)

    def draw_noise_into(self, buf):
        """Fill ``buf`` [n, A] with this step's sampling noise (one draw for the whole env batch)."""
        if hasattr(self.noise_fn, "inplace"):
            self.noise_fn.inplace(buf)
        else:
            buf.copy_(self.noise_fn(buf.shape[0], buf.shape[1], buf.device))

    def sample_into(self, obs, actions_out, logprobs_out, values_out, noise=None):
        """Rollout step: forward + sample, writing straight into the rollout slots (ppo.py:197-202).
        ``noise``: pre-drawn rows of the step's noise tensor (chunked H2D/compute pipeline)."""
        logits, value = self._forward_heads(obs)
        n, A = logits.shape
        q = noise if noise is not None else self.noise_fn(n, A, logits.device)
        ops.categorical_sample(logits, q, value, out=(actions_out, logprobs_out, None, values_out))

    def loss_backward(self, policy_out, value, mb_inds, b, a, stats_row, scratch):
        """Minibatch loss (+ its gradient) and the network backward (ppo.py:251-288)."""
        M = policy_out.shape[0]
        if scratch.get("M") != M:
            scratch["M"] = M
            scratch["dhead"], scratch["dl"], scratch["dv"] = self.alloc_head_grad(M, policy_out.device)
        ops.ppo_loss(policy_out, value, mb_inds, b["actions"], b["logprobs"], b["advantages"], b["returns"], b["values"],
                     a.clip_coef, a.ent_coef, a.vf_coef, a.norm_adv, a.clip_vloss,
                     dlogits=scratch["dl"], dvalue=scratch["dv"], stats=stats_row)
        self.backward(scratch["dhead"])

    # -- reference API ---------------------------------------------------------
    def get_value(self, x):
        self.flat
        _, value = self._forward_heads(x)
        return value.reshape(-1, 1).clone() if not value.is_contiguous() else value.reshape(-1, 1)

    def get_action_and_value(self, x, action=None):
        self.flat
        logits, value = self._forward_heads(x)
        n, A = logits.shape
        if action is None:
            q = self.noise_fn(n, A, logits.device)
            action, logprob, entropy, v = ops.categorical_sample(logits, q, value)
        else:
            logprob, entropy = ops.categorical_eval(logits, action)
            v = value.clone() if not value.is_contiguous() else value
        return action, logprob, entropy, v.reshape(-1, 1)


class NatureCNNAgent(KernelAgent):
    """NatureCNN actor-critic (reference: cleanrl/ppo_atari_envpool.py:123-149)."""

    def __init__(self, envs):
        super().__init__()
        c, h, w = envs.single_observation_space.shape
        assert (c, h, w) == (4, 84, 84), "NatureCNN geometry is 4x84x84"
        trunk = []
        for cin, cout, k, s in ((4, 32, 8, 4), (32, 64, 4, 2), (64, 64, 3, 1)):
            trunk += [layer_init(nn.Conv2d(cin, cout, k, stride=s)), nn.ReLU()]
        trunk += [nn.Flatten(), layer_init(nn.Linear(64 * 7 * 7, 512)), nn.ReLU()]
        self.network = nn.Sequential(*trunk)
        self.actor = layer_init(nn.Linear(512, envs.single_action_space.n), std=0.01)
        self.critic = layer_init(nn.Linear(512, 1), std=1)
        self.num_actions = int(envs.single_action_space.n)

    def _param_order(self):
        net = [p for m in self.network for p in m.parameters()]
        # both heads adjacent => one [A+1, 512] GEMM operand and one [A+1] bias
        return net + [self.actor.weight, self.critic.weight, self.actor.bias, self.critic.bias]

    def _build_plan(self):
        f = self._flat
        A = self.num_actions
        wa, ga = f.view_of(self.actor.weight)
        ba, gba = f.view_of(self.actor.bias)
        off_w = (wa.data_ptr() - f.flat.data_ptr()) // 4
        off_b = (ba.data_ptr() - f.flat.data_ptr()) // 4
        self._head_w = f.flat[off_w:off_w + (A + 1) * 512].view(A + 1, 512)
        self._head_b = f.flat[off_b:off_b + A + 1]
        self._head_dw = f.grad[off_w:off_w + (A + 1) * 512].view(A + 1, 512)
        self._head_db = f.grad[off_b:off_b + A + 1]
        n = self.network
        self.trunk = nets.Chain([
            nets.Conv(n[0], "relu", in_div=255.0), nets.Conv(n[2], "relu"), nets.Conv(n[4], "relu"),
            nets.Linear(n[7], "relu")])
        self.head = nets.Linear(None, None, self._head_w, self._head_b, self._head_dw, self._head_db)
        self._tc = None
        self._tc_dirty = True

    # -- bf16 tensor-core plan ("--precision bf16") ------------------------------
    precision = "fp32"

    def params_updated(self):
        """Call after the optimiser changed the flat parameters: the packed bf16 operands are stale."""
        self._tc_dirty = True

    def _tc_plan(self):
        f = self._flat
        if self._tc is None:
            assert f.flat.numel() >= ops._lib.load().b200rl_naturecnn_param_count(self.num_actions)
            self._tc = ops.NatureCNNBf16(self.num_actions, f.flat.device)
        if self._tc_dirty:
            self._tc.pack(f.flat)
            self._tc_dirty = False
        return self._tc

    def load_state_dict(self, *a, **k):
        out = super().load_state_dict(*a, **k)
        self._tc_dirty = True
        return out

    def pin_workspaces(self):
        """A CUDA graph captured by the engine holds raw pointers into the activation workspaces: never evict them."""
        if self._tc is not None:
            self._tc.pin()

    def _forward_heads(self, x, rows=None, keep=False, aux=None):
        if self.precision == "bf16":
            if x.dtype not in (torch.uint8, torch.bfloat16):
                x = x.to(torch.uint8)       # frames are integers 0..255 (reference passes them as fp32)
            tc = self._tc_plan()
            out = tc.forward(x.contiguous(), rows, self._flat.flat)
            if keep:
                self._tc_obs, self._tc_rows, self._tc_aux = x, rows, aux
            A = self.num_actions
            return out[:, :A], out[:, A]
        if x.dtype not in (torch.uint8, torch.float32):
            x = x.float()
        hidden = self.trunk.fwd(x.contiguous(), rows=rows, keep=keep)
        out = self.head.fwd(hidden)
        if keep:
            self._hidden = hidden
        A = self.num_actions
        return out[:, :A], out[:, A]

    def rollout_step_into(self, frames, slot_rm, slot_cm, actions_out, logprobs_out, values_out, noise=None):
        """Rollout step of the bf16 path on the uint8 rollout layout: ``frames`` (uint8 [n,4,84,84], or None when
        ``slot_rm`` is already written) -> both slot orientations + forward + sample in one native call.  Same results
        as ``frames_to_s2d_u8`` followed by ``sample_into`` on the slot."""
        n, A = slot_rm.shape[0], self.num_actions
        q = noise if noise is not None else self.noise_fn(n, A, slot_rm.device)
        self._tc_plan().rollout_step(frames, slot_rm, slot_cm, self._flat.flat, q, actions_out, logprobs_out, values_out)

    def forward_train(self, b_obs, mb_inds, aux=None):
        """Minibatch forward with fused row gather (b_obs[mb_inds] never materialised); keeps activations.
        ``aux``: channel-major copy of a uint8 space-to-depth rollout (consumed by the conv1 weight gradient)."""
        self.flat
        return self._forward_heads(b_obs, rows=mb_inds, keep=True, aux=aux)

    def alloc_head_grad(self, M, device):
        A = self.num_actions
        d = torch.empty(M, A + 1, dtype=torch.float32, device=device)
        return d, d[:, :A], d[:, A]

    def grad_tail(self):
        """(offset, event): ``flat.grad[offset:]`` (fc + heads, 95 % of the vector) is final when ``event`` fires in the
        middle of ``backward`` -- lets the engine overlap the DP exchange of the tail with the conv backward.  None on
        the fp32 path (layer-by-layer backward finishes the first layers' gradients last anyway, but records no event)."""
        if self.precision != "bf16":
            return None
        if getattr(self, "_tail_event", None) is None:
            self._tail_event = torch.cuda.Event()
            self._tail_event.record()                      # materialise the cudaEvent_t handle
        return self._tc_plan().grad_tail_offset(), self._tail_event

    def backward(self, dhead):
        """dhead [M, A+1] = [dlogits | dvalue]; fills the flat gradient buffer."""
        if self.precision == "bf16":
            self._tc.backward(self._tc_obs, self._tc_rows, self._flat.flat, dhead, self._flat.grad,
                              tail_event=getattr(self, "_tail_event", None), obs_aux=getattr(self, "_tc_aux", None))
            self._tc_obs = self._tc_rows = self._tc_aux = None
            return
        hidden = self._hidden
        self.head.bwd_weight(hidden, dhead)
        dh = self.head.bwd_data(dhead, hidden, "relu")
        self.trunk.bwd(dh)
        self._hidden = None


class MLPAgent(KernelAgent):
    """Two 64-wide tanh MLPs, discrete actions (reference: cleanrl/ppo.py:100-126)."""

    def __init__(self, envs):
        super().__init__()
        d = int(np.array(envs.single_observation_space.shape).prod())
        A = int(envs.single_action_space.n)
        self.critic = nn.Sequential(layer_init(nn.Linear(d, 64)), nn.Tanh(), layer_init(nn.Linear(64, 64)), nn.Tanh(),
                                    layer_init(nn.Linear(64, 1), std=1.0))
        self.actor = nn.Sequential(layer_init(nn.Linear(d, 64)), nn.Tanh(), layer_init(nn.Linear(64, 64)), nn.Tanh(),
                                   layer_init(nn.Linear(64, A), std=0.01))
        self.num_actions = A

    def _build_plan(self):
        mk = lambda seq: nets.Chain([nets.Linear(seq[0], "tanh"), nets.Linear(seq[2], "tanh"), nets.Linear(seq[4], None)])
        self.c_chain, self.a_chain = mk(self.critic), mk(self.actor)

    def _forward_heads(self, x, rows=None, keep=False):
        x = x.float() if x.dtype != torch.float32 else x
        x = x.reshape(x.shape[0], -1).contiguous()
        logits = self.a_chain.fwd(x, rows=rows, keep=keep)
        value = self.c_chain.fwd(x, rows=rows, keep=keep)
        return logits, value[:, 0]

    def forward_train(self, b_obs, mb_inds):
        self.flat
        return self._forward_heads(b_obs, rows=mb_inds, keep=True)

    def alloc_head_grad(self, M, device):
        dl = torch.empty(M, self.num_actions, dtype=torch.float32, device=device)
        dv = torch.empty(M, 1, dtype=torch.float32, device=device)
        return (dl, dv), dl, dv[:, 0]

    def backward(self, dhead):
        dl, dv = dhead
        self.a_chain.bwd(dl)
        self.c_chain.bwd(dv)


class LSTMAgent(KernelAgent):
    """Recurrent actor-critic (reference: cleanrl/ppo_atari_lstm.py:117-160): NatureCNN trunk over ONE grayscale frame,
    ``nn.LSTM(512, 128)`` with the state reset by ``(1 - done)`` before every step, ``actor`` / ``critic`` on the LSTM
    output.  Same module names / ``state_dict`` keys (``network.*``, ``lstm.weight_ih_l0`` ..., ``actor.*``, ``critic.*``),
    same initialisation order (orthogonal_ on the two LSTM weight matrices with gain 1, biases zero).

    Execution: fp32 kernels of libb200rl, no autograd.  The trunk and the input-gate GEMM ``x W_ih^T + b_ih`` run once over
    ALL steps of a sequence; per step there is one small GEMM ``h' W_hh^T + b_hh`` and one fused cell kernel.  The backward
    pass is explicit back-propagation through time (one cell-backward kernel + one ``dgates W_hh`` GEMM per step), after
    which the weight gradients of both LSTM matrices and of the trunk are single GEMMs over the whole sequence."""

    def __init__(self, envs):
        super().__init__()
        c, h, w = envs.single_observation_space.shape
        assert (h, w) == (84, 84), "NatureCNN trunk geometry is 84x84"
        trunk = []
        for cin, cout, k, s in ((c, 32, 8, 4), (32, 64, 4, 2), (64, 64, 3, 1)):
            trunk += [layer_init(nn.Conv2d(cin, cout, k, stride=s)), nn.ReLU()]
        trunk += [nn.Flatten(), layer_init(nn.Linear(64 * 7 * 7, 512)), nn.ReLU()]
        self.network = nn.Sequential(*trunk)
        self.lstm = nn.LSTM(512, 128)
        for name, param in self.lstm.named_parameters():
            if "bias" in name:
                nn.init.constant_(param, 0)
            elif "weight" in name:
                nn.init.orthogonal_(param, 1.0)
        self.actor = layer_init(nn.Linear(128, envs.single_action_space.n), std=0.01)
        self.critic = layer_init(nn.Linear(128, 1), std=1)
        self.num_actions = int(envs.single_action_space.n)
        self.hidden_size = 128

    def _param_order(self):
        net = [p for m in self.network for p in m.parameters()]
        return net + list(self.lstm.parameters()) + [self.actor.weight, self.critic.weight, self.actor.bias, self.critic.bias]

    def _build_plan(self):
        f = self._flat
        A, H = self.num_actions, self.hidden_size
        wa, _ = f.view_of(self.actor.weight)
        ba, _ = f.view_of(self.actor.bias)
        off_w = (wa.data_ptr() - f.flat.data_ptr()) // 4
        off_b = (ba.data_ptr() - f.flat.data_ptr()) // 4
        head_w = f.flat[off_w:off_w + (A + 1) * H].view(A + 1, H)
        head_b = f.flat[off_b:off_b + A + 1]
        head_dw = f.grad[off_w:off_w + (A + 1) * H].view(A + 1, H)
        head_db = f.grad[off_b:off_b + A + 1]
        n = self.network
        self.trunk = nets.Chain([nets.Conv(n[0], "relu", in_div=255.0), nets.Conv(n[2], "relu"), nets.Conv(n[4], "relu"),
                                 nets.Linear(n[7], "relu")])
        self.head = nets.Linear(None, None, head_w, head_b, head_dw, head_db)
        L = self.lstm
        self.l_ih = nets.Linear(None, None, L.weight_ih_l0.data, L.bias_ih_l0.data, L.weight_ih_l0.grad, L.bias_ih_l0.grad)
        self.l_hh = nets.Linear(None, None, L.weight_hh_l0.data, L.bias_hh_l0.data, L.weight_hh_l0.grad, L.bias_hh_l0.grad)

    graph_capturable = False

    # ------------------------------------------------------------------ forward
    def get_states(self, x, lstm_state, done, rows=None, keep=False):
        """hidden [S*n, H], (h_S, c_S): ``x`` = S*n frames (or ``rows`` gathering them from a larger buffer), time-major."""
        self.flat
        H = self.hidden_size
        h, c = lstm_state[0].reshape(-1, H).contiguous(), lstm_state[1].reshape(-1, H).contiguous()
        n = h.shape[0]
        if x.dtype not in (torch.uint8, torch.float32):
            x = x.float()
        feats = self.trunk.fwd(x.contiguous(), rows=rows, keep=keep)            # [S*n, 512], post-ReLU
        total = feats.shape[0]
        assert total % n == 0, "the sequence batch must be steps x envs"
        S = total // n
        dev = feats.device
        done = done.reshape(S, n).to(torch.float32).contiguous()
        gx = self.l_ih.fwd(feats)                                               # [S*n, 4H] for every step at once
        hidden = torch.empty(S, n, H, dtype=torch.float32, device=dev)
        hm = torch.empty(S, n, H, dtype=torch.float32, device=dev)
        cm = torch.empty(S, n, H, dtype=torch.float32, device=dev)
        save = torch.empty(S, n, 5 * H, dtype=torch.float32, device=dev) if keep else None
        c_cur = torch.empty(n, H, dtype=torch.float32, device=dev)
        for t in range(S):
            ops.lstm_mask_state(h, c, done[t], out=(hm[t], cm[t]))
            gh = self.l_hh.fwd(hm[t])
            ops.lstm_cell_fwd(gx[t * n:(t + 1) * n], gh, cm[t], hidden[t], c_cur, save[t] if keep else None)
            h, c = hidden[t], c_cur
            if t + 1 < S:
                c_cur = torch.empty(n, H, dtype=torch.float32, device=dev)
        if keep:
            self._seq = dict(feats=feats, hidden=hidden, hm=hm, cm=cm, save=save, done=done, S=S, n=n)
        return hidden.view(S * n, H), (h.reshape(1, n, H).clone(), c.reshape(1, n, H).clone())

    def _heads(self, hidden):
        out = self.head.fwd(hidden)
        A = self.num_actions
        return out[:, :A], out[:, A]

    def get_value(self, x, lstm_state, done):
        hidden, _ = self.get_states(x, lstm_state, done)
        _, value = self._heads(hidden)
        return value.reshape(-1, 1).clone()

    def get_action_and_value(self, x, lstm_state, done, action=None, rows=None, keep=False):
        hidden, lstm_state = self.get_states(x, lstm_state, done, rows=rows, keep=keep)
        logits, value = self._heads(hidden)
        if keep:
            self._seq["logits"], self._seq["value"] = logits, value
        m, A = logits.shape
        if action is None:
            q = self.noise_fn(m, A, logits.device)
            action, logprob, entropy, v = ops.categorical_sample(logits, q, value)
        else:
            logprob, entropy = ops.categorical_eval(logits, action)
            v = value.clone()
        return action, logprob, entropy, v.reshape(-1, 1), lstm_state

    def forward_train(self, b_obs, mb_inds, lstm_state, b_dones):
        """Minibatch forward over whole env sequences (mb_inds time-major: step t of every env of the minibatch, then
        step t+1, ... as cleanrl/ppo_atari_lstm.py:303), activations kept for ``backward``."""
        done = b_dones.reshape(-1)[mb_inds]
        hidden, _ = self.get_states(b_obs, lstm_state, done, rows=mb_inds, keep=True)
        return self._heads(hidden)

    def alloc_head_grad(self, M, device):
        A = self.num_actions
        d = torch.empty(M, A + 1, dtype=torch.float32, device=device)
        return d, d[:, :A], d[:, A]

    # ----------------------------------------------------------------- backward
    def backward(self, dhead):
        q = self._seq
        S, n, H = q["S"], q["n"], self.hidden_size
        hidden = q["hidden"].view(S * n, H)
        self.head.bwd_weight(hidden, dhead)
        dh_heads = self.head.bwd_data(dhead, None, None).view(S, n, H)
        dev = dhead.device
        dgates = torch.empty(S, n, 4 * H, dtype=torch.float32, device=dev)
        dc_a = torch.empty(n, H, dtype=torch.float32, device=dev)
        dc_b = torch.empty(n, H, dtype=torch.float32, device=dev)
        dh_rec, dc_rec = None, None
        for t in reversed(range(S)):
            ops.lstm_cell_bwd(dh_heads[t], dh_rec, q["done"][t + 1] if t + 1 < S else None, dc_rec, q["save"][t], q["cm"][t],
                              q["done"][t], dgates[t], dc_a)
            dc_rec, dc_a, dc_b = dc_a, dc_b, dc_a
            if t > 0:
                dh_rec = self.l_hh.bwd_data(dgates[t], None, None)             # dgates_t W_hh -> d h'_{t-1} (masked at t-1's kernel)
        dg = dgates.view(S * n, 4 * H)
        self.l_hh.bwd_weight(q["hm"].view(S * n, H), dg)
        self.l_ih.bwd_weight(q["feats"], dg)
        dfeats = self.l_ih.bwd_data(dg, q["feats"], "relu")
        self.trunk.bwd(dfeats)
        self._seq = None


class ResidualBlock(nn.Module):
    """Parameter container with the reference's names (cleanrl/ppo_procgen.py:89-102); executed by ImpalaAgent."""

    def __init__(self, channels):
        super().__init__()
        self.conv0 = nn.Conv2d(in_channels=channels, out_channels=channels, kernel_size=3, padding=1)
        self.conv1 = nn.Conv2d(in_channels=channels, out_channels=channels, kernel_size=3, padding=1)


class ConvSequence(nn.Module):
    """cleanrl/ppo_procgen.py:105-124: conv3x3 -> max_pool(3, stride 2, padding 1) -> two residual blocks."""

    def __init__(self, input_shape, out_channels):
        super().__init__()
        self._input_shape = input_shape
        self._out_channels = out_channels
        self.conv = nn.Conv2d(in_channels=self._input_shape[0], out_channels=self._out_channels, kernel_size=3, padding=1)
        self.res_block0 = ResidualBlock(self._out_channels)
        self.res_block1 = ResidualBlock(self._out_channels)

    def get_output_shape(self):
        _c, h, w = self._input_shape
        return (self._out_channels, (h + 1) // 2, (w + 1) // 2)


class ImpalaAgent(KernelAgent):
    """IMPALA-CNN actor-critic (reference: cleanrl/ppo_procgen.py:89-150): three ConvSequences (16, 32, 32 channels),
    Flatten, ReLU, Linear(2048 -> 256), ReLU, ``actor`` / ``critic``.  Same module tree (``network.{0,1,2}.conv``,
    ``network.{0,1,2}.res_block{0,1}.conv{0,1}``, ``network.5``), same construction order, torch's default initialisation
    for the trunk (the reference only ``layer_init``s the heads), so a seed yields the reference's weights and
    ``state_dict`` files interchange.  Frames arrive NHWC uint8 ([n, 64, 64, 3]) and are permuted on the device.

    Execution: fp32 kernels of libb200rl (padded 3x3 convolutions, max-pool with arg-max, ReLU / add glue), explicit
    backward in reverse order; no autograd, no cuDNN."""

    def __init__(self, envs):
        super().__init__()
        h, w, c = envs.single_observation_space.shape
        shape = (c, h, w)
        conv_seqs = []
        for out_channels in [16, 32, 32]:
            conv_seq = ConvSequence(shape, out_channels)
            shape = conv_seq.get_output_shape()
            conv_seqs.append(conv_seq)
        conv_seqs += [nn.Flatten(), nn.ReLU(),
                      nn.Linear(in_features=shape[0] * shape[1] * shape[2], out_features=256), nn.ReLU()]
        self.network = nn.Sequential(*conv_seqs)
        self.actor = layer_init(nn.Linear(256, envs.single_action_space.n), std=0.01)
        self.critic = layer_init(nn.Linear(256, 1), std=1)
        self.num_actions = int(envs.single_action_space.n)
        self._feat_shape = shape

    graph_capturable = False

    def _param_order(self):
        net = [p for p in self.network.parameters()]
        return net + [self.actor.weight, self.critic.weight, self.actor.bias, self.critic.bias]

    def _build_plan(self):
        f = self._flat
        A = self.num_actions
        wa, _ = f.view_of(self.actor.weight)
        ba, _ = f.view_of(self.actor.bias)
        off_w = (wa.data_ptr() - f.flat.data_ptr()) // 4
        off_b = (ba.data_ptr() - f.flat.data_ptr()) // 4
        self.head = nets.Linear(None, None, f.flat[off_w:off_w + (A + 1) * 256].view(A + 1, 256), f.flat[off_b:off_b + A + 1],
                                f.grad[off_w:off_w + (A + 1) * 256].view(A + 1, 256), f.grad[off_b:off_b + A + 1])
        self.fc = nets.Linear(self.network[5], "relu")
        self.seqs = []
        for i in range(3):
            q = self.network[i]
            self.seqs.append(dict(conv=nets.Conv(q.conv, None, in_div=255.0 if i == 0 else 1.0),
                                  blocks=[(nets.Conv(b.conv0, "relu"), nets.Conv(b.conv1, None))
                                          for b in (q.res_block0, q.res_block1)]))

    # ------------------------------------------------------------------ forward
    def _forward_heads(self, x, rows=None, keep=False):
        if x.dtype != torch.uint8:
            x = x.to(torch.uint8)          # frames are integers 0..255 (the reference passes them as fp32)
        x = ops.nhwc_to_nchw_u8(x.contiguous(), rows)          # [n, 3, 64, 64] uint8; /255 inside the first convolution
        saved = []
        h = x
        for s in self.seqs:
            c = s["conv"].fwd(h)                               # conv, no activation
            p, arg = ops.maxpool3s2_fwd(c)
            rec = dict(x=h, c_hw=tuple(c.shape[-2:]), arg=arg, blocks=[])
            b = p
            for conv0, conv1 in s["blocks"]:
                r0 = ops.relu(b)                               # x -> relu -> conv0 -> relu -> conv1 -> + x
                y0 = conv0.fwd(r0)                             # relu fused on the output (the next op is a relu)
                c1 = conv1.fwd(y0)
                out = ops.add(c1, b)
                rec["blocks"].append((r0, y0))
                b = out
            saved.append(rec)
            h = b
        flat = h.reshape(h.shape[0], -1)
        h0 = ops.relu(flat)                                    # Flatten, ReLU
        hid = self.fc.fwd(h0)                                  # Linear + ReLU
        out = self.head.fwd(hid)
        if keep:
            self._saved = dict(seqs=saved, h0=h0, hid=hid, last_shape=tuple(h.shape))
        A = self.num_actions
        return out[:, :A], out[:, A]

    def forward_train(self, b_obs, mb_inds):
        self.flat
        return self._forward_heads(b_obs, rows=mb_inds, keep=True)

    def alloc_head_grad(self, M, device):
        A = self.num_actions
        d = torch.empty(M, A + 1, dtype=torch.float32, device=device)
        return d, d[:, :A], d[:, A]

    # ----------------------------------------------------------------- backward
    def backward(self, dhead):
        q = self._saved
        self.head.bwd_weight(q["hid"], dhead)
        d_hid = self.head.bwd_data(dhead, q["hid"], "relu")                    # through the ReLU after the Linear
        self.fc.bwd_weight(q["h0"], d_hid)
        d = self.fc.bwd_data(d_hid, q["h0"], "relu").view(q["last_shape"])     # through the ReLU after Flatten
        for si in (2, 1, 0):
            s, rec = self.seqs[si], q["seqs"][si]
            for (conv0, conv1), (r0, y0) in zip(reversed(s["blocks"]), reversed(rec["blocks"])):
                conv1.bwd_weight(y0, d)
                dy0 = conv1.bwd_data(d, y0, "relu")                            # * (y0 > 0)
                conv0.bwd_weight(r0, dy0)
                d_in = conv0.bwd_data(dy0, None, None, in_hw=tuple(r0.shape[-2:]))
                d = ops.relu_bwd(d_in, r0, extra=d)                            # * (x > 0) + skip connection
            d_c = ops.maxpool3s2_bwd(d, rec["arg"], rec["c_hw"])
            s["conv"].bwd_weight(rec["x"], d_c)
            if si > 0:
                d = s["conv"].bwd_data(d_c, None, None, in_hw=tuple(rec["x"].shape[-2:]))
        self._saved = None


def _normal_noise(n, D, device):
    # what Normal(mean, std).sample() == torch.normal(mean, std) consumes: one N(0,1) per element
    return torch.randn(n, D, dtype=torch.float32, device=device)


_normal_noise.graph_safe = True
_normal_noise.inplace = lambda buf: buf.normal_(0, 1)


class ContinuousMLPAgent(KernelAgent):
    """Gaussian-policy MLP agent (reference: cleanrl/ppo_continuous_action.py:112-141): ``critic`` and
    ``actor_mean`` Sequentials plus the state-independent ``actor_logstd`` parameter [1, D]."""

    def __init__(self, envs):
        super().__init__()
        d = int(np.array(envs.single_observation_space.shape).prod())
        D = int(np.prod(envs.single_action_space.shape))
        self.critic = nn.Sequential(layer_init(nn.Linear(d, 64)), nn.Tanh(), layer_init(nn.Linear(64, 64)), nn.Tanh(),
                                    layer_init(nn.Linear(64, 1), std=1.0))
        self.actor_mean = nn.Sequential(layer_init(nn.Linear(d, 64)), nn.Tanh(), layer_init(nn.Linear(64, 64)), nn.Tanh(),
                                        layer_init(nn.Linear(64, D), std=0.01))
        self.actor_logstd = nn.Parameter(torch.zeros(1, D))
        self.action_dim = D
        self.noise_fn = _normal_noise

    def _build_plan(self):
        mk = lambda seq: nets.Chain([nets.Linear(seq[0], "tanh"), nets.Linear(seq[2], "tanh"), nets.Linear(seq[4], None)])
        self.c_chain, self.a_chain = mk(self.critic), mk(self.actor_mean)

    def _forward_heads(self, x, rows=None, keep=False):
        x = x.float() if x.dtype != torch.float32 else x
        x = x.reshape(x.shape[0], -1).contiguous()
        mean = self.a_chain.fwd(x, rows=rows, keep=keep)
        value = self.c_chain.fwd(x, rows=rows, keep=keep)
        return mean, value[:, 0]

    def forward_train(self, b_obs, mb_inds):
        self.flat
        return self._forward_heads(b_obs, rows=mb_inds, keep=True)

    def _logstd(self):
        return self.actor_logstd.data.view(-1)

    def noise_shape(self, n):
        return (n, self.action_dim)

    def sample_into(self, obs, actions_out, logprobs_out, values_out, noise=None):
        mean, value = self._forward_heads(obs)
        n, D = mean.shape
        eps = noise if noise is not None else self.noise_fn(n, D, mean.device)
        ops.gaussian_sample(mean, self._logstd(), eps, value, out=(actions_out, logprobs_out, None, values_out))

    def loss_backward(self, policy_out, value, mb_inds, b, a, stats_row, scratch):
        M, D = policy_out.shape
        dev = policy_out.device
        if scratch.get("M") != M:
            scratch["M"] = M
            scratch["dmean"] = torch.empty(M, D, dtype=torch.float32, device=dev)
            scratch["dv"] = torch.empty(M, 1, dtype=torch.float32, device=dev)
        ops.ppo_loss_gaussian(policy_out, self._logstd(), value, mb_inds, b["actions"], b["logprobs"], b["advantages"],
                              b["returns"], b["values"], a.clip_coef, a.ent_coef, a.vf_coef, a.norm_adv, a.clip_vloss,
                              dmean=scratch["dmean"], dlogstd=self.actor_logstd.grad.view(-1), dvalue=scratch["dv"][:, 0],
                              stats=stats_row)
        self.a_chain.bwd(scratch["dmean"])
        self.c_chain.bwd(scratch["dv"])

    def get_action_and_value(self, x, action=None):
        self.flat
        mean, value = self._forward_heads(x)
        n, D = mean.shape
        if action is None:
            eps = self.noise_fn(n, D, mean.device)
            action, logprob, entropy, v = ops.gaussian_sample(mean, self._logstd(), eps, value)
        else:
            logprob, entropy = ops.gaussian_eval(mean, self._logstd(), action)
            v = value.clone() if not value.is_contiguous() else value
        return action, logprob, entropy, v.reshape(-1, 1)


class QNetworkAgent(nn.Module):
    """DQN Q-network (reference: cleanrl/dqn_atari.py:108-125): NatureCNN trunk + Linear(512, A), default torch
    initialisation, ``forward(x)`` -> Q-values [n, A]; state_dict keys ``network.{0,2,4,7,9}.*``."""

    def __init__(self, env):
        super().__init__()
        A = int(env.single_action_space.n)
        self.network = nn.Sequential(
            nn.Conv2d(4, 32, 8, stride=4), nn.ReLU(), nn.Conv2d(32, 64, 4, stride=2), nn.ReLU(),
            nn.Conv2d(64, 64, 3, stride=1), nn.ReLU(), nn.Flatten(), nn.Linear(3136, 512), nn.ReLU(), nn.Linear(512, A))
        self.num_actions = A
        self.precision = "fp32"
        self._flat = None
        self._tc = None
        self._tc_dirty = True

    def bind(self):
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("cleanrl_b200 agents execute on CUDA only (libb200rl kernels); "
                               f"parameters are on {dev}. There is no CPU fallback.")
        self._flat = nets.FlatParams(list(self.parameters()), dev)   # natural order == libb200rl NatureCNN order
        n = self.network
        self.chain = nets.Chain([nets.Conv(n[0], "relu", in_div=255.0), nets.Conv(n[2], "relu"), nets.Conv(n[4], "relu"),
                                 nets.Linear(n[7], "relu"), nets.Linear(n[9], None)])
        return self._flat

    @property
    def flat(self):
        if self._flat is None or self._flat.flat.device != next(self.parameters()).device:
            self.bind()
        return self._flat

    def params_updated(self):
        self._tc_dirty = True

    def load_state_dict(self, *a, **k):
        out = super().load_state_dict(*a, **k)
        self._tc_dirty = True
        return out

    def _plan(self):
        f = self.flat
        if self._tc is None:
            self._tc = ops.NatureCNNBf16(self.num_actions - 1, f.flat.device)   # heads = (A-1) + 1 = A outputs
        if self._tc_dirty:
            self._tc.pack(f.flat)
            self._tc_dirty = False
        return self._tc

    def q_values(self, frames, rows=None, keep=False):
        """Q(s, .) for frames[rows] (uint8 [*,4,84,84]; rows gathers without materialising)."""
        self.flat
        if frames.dtype != torch.uint8:
            frames = frames.to(torch.uint8)
        if self.precision == "bf16":
            out = self._plan().forward(frames.contiguous(), rows, self._flat.flat)
            if keep:
                self._saved = (frames, rows)
            return out
        return self.chain.fwd(frames.contiguous(), rows=rows, keep=keep)

    def forward(self, x):
        return self.q_values(x)

    def backward(self, dq):
        if self.precision == "bf16":
            frames, rows = self._saved
            self._tc.backward(frames, rows, self._flat.flat, dq, self._flat.grad)
            self._saved = None
        else:
            self.chain.bwd(dq)


def dqn_update(q_network, target_network, ring, batch, gamma, lr, huber=False, stats=None):
    """One TD update (reference: dqn_atari.py:219-235): target forward, online forward, fused TD loss + dL/dQ,
    hand-written backward, Adam (torch defaults eps=1e-8, no gradient clipping)."""
    frames = ring.frames
    with torch.no_grad():
        qt = target_network.q_values(frames, rows=batch["next_rows"])
        q = q_network.q_values(frames, rows=batch["rows"], keep=True)
        stats, dq = ops.dqn_td_loss(q, qt, batch["actions"], batch["rewards"], batch["dones"], gamma, huber=huber, stats=stats)
        q_network.backward(dq)
        f = q_network.flat
        f.step += 1
        ops.clip_adam(f.flat, f.grad, f.exp_avg, f.exp_avg_sq, f.step, lr, eps=1e-8, max_norm=None)
        q_network.params_updated()
    return stats


def dqn_sync_target(q_network, target_network, tau=1.0):
    """dqn_atari.py:238-242: target <- tau * online + (1 - tau) * target (flat buffers, one fused axpby)."""
    t, q = target_network.flat.flat, q_network.flat.flat
    if tau == 1.0:
        t.copy_(q)
    else:
        t.mul_(1.0 - tau).add_(q, alpha=tau)
    target_network.params_updated()
