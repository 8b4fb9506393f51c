"""Generate tests/golden/*.npz from the UNMODIFIED reference (build container only).

    python -m oracle.make_golden

Each fixture records what the reference script computed on CPU for a small,
seeded configuration of the synthetic envs; the GPU box (which has no
/root/reference) replays the same configuration through the CUDA path and
compares.  TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import ast
import hashlib
import json
import sys
from pathlib import Path

import numpy as np

from oracle.ref_harness import REFERENCE_ROOT, run_reference

OUT = Path(__file__).resolve().parent.parent / "tests" / "golden"


def _stack(recs, key):
    return np.stack([r[key] for r in recs])


def atari_envpool(name, argv, n_iter, script="ppo_atari_envpool.py", gymnasium_kind="atari"):
    """cleanrl/ppo_atari_envpool.py (envpool/gym-0.23 API), cleanrl/ppo_atari.py (gymnasium API) or
    cleanrl/ppo_atari_lstm.py (gymnasium API, one grayscale frame: kind "atari1") on the Breakout-shaped synthetic env."""
    rec, g = run_reference(script, argv, atari_mode="fresh", gymnasium_kind=gymnasium_kind)
    assert len(rec.iterations) == n_iter
    out = {"argv": np.array(argv)}
    for k in ("actions", "logprobs", "rewards", "dones", "values", "advantages", "returns", "next_value", "next_done",
              "param_sums", "param_abs_sums"):
        out[k] = _stack(rec.iterations, k)
    for k in ("pg_loss", "v_loss", "entropy_loss", "old_approx_kl", "approx_kl", "loss", "clipfrac", "lr",
              "grad_norm_postclip"):
        out["upd_" + k] = np.array([u[k] for u in rec.updates])
    out["upd_param_sums"] = _stack(rec.updates, "param_sums")
    out["upd_mb_inds_head"] = _stack(rec.updates, "mb_inds_head")
    out["shuffles"] = np.stack(rec.shuffles)
    tags = sorted({t for t, _, _ in rec.scalars})
    for t in tags:
        vals = [(s, v) for tt, v, s in rec.scalars if tt == t]
        out["tb/" + t] = np.array(vals, dtype=np.float64)
    np.savez_compressed(OUT / name, **out)
    print("wrote", name, {k: v.shape for k, v in out.items() if hasattr(v, "shape")})


def atari_envpool_full(name, argv):
    """The HEADLINE configuration (BASELINE.json configs[1]: num_envs=1024, num_steps=128, minibatch 32 768), one
    iteration of the unmodified cleanrl/ppo_atari_envpool.py on the Breakout-shaped synthetic env.  Integer-valued
    tensors are stored narrow (actions int8, rewards int8, dones uint8) to keep the fixture at a few MB."""
    rec, g = run_reference("ppo_atari_envpool.py", argv, atari_mode="fresh", gymnasium_kind="atari")
    assert len(rec.iterations) == 1
    it = rec.iterations[0]
    out = {"argv": np.array(argv)}
    assert np.array_equal(it["actions"], it["actions"].astype(np.int8)) and np.array_equal(it["rewards"], it["rewards"].astype(np.int8))
    out["actions"] = it["actions"].astype(np.int8)[None]
    out["rewards"] = it["rewards"].astype(np.int8)[None]
    out["dones"] = it["dones"].astype(np.uint8)[None]
    for k in ("logprobs", "values", "advantages", "returns", "next_value", "next_done", "param_sums", "param_abs_sums"):
        out[k] = it[k][None]
    for k in ("pg_loss", "v_loss", "entropy_loss", "old_approx_kl", "approx_kl", "loss", "clipfrac", "lr",
              "grad_norm_postclip"):
        out["upd_" + k] = np.array([u[k] for u in rec.updates])
    out["upd_param_sums"] = _stack(rec.updates, "param_sums")
    out["upd_mb_inds_head"] = _stack(rec.updates, "mb_inds_head")
    out["shuffles"] = np.stack(rec.shuffles)
    for t in sorted({t for t, _, _ in rec.scalars}):
        out["tb/" + t] = np.array([(s, v) for tt, v, s in rec.scalars if tt == t], dtype=np.float64)
    np.savez_compressed(OUT / name, **out)
    print("wrote", name, {k: v.shape for k, v in out.items() if hasattr(v, "shape")})


def mlp_ppo(name, argv):
    """cleanrl/ppo.py with the CartPole-shaped synthetic env: per-update tensors for loss/Adam oracles."""
    rec, g = run_reference("ppo.py", argv, gymnasium_kind="discrete", keep_params=True)
    out = {"argv": np.array(argv)}
    for k in ("actions", "logprobs", "rewards", "dones", "values", "advantages", "returns", "next_value", "next_done"):
        out[k] = _stack(rec.iterations, k)
    ups = rec.updates[:6]
    for k in ("pg_loss", "v_loss", "entropy_loss", "old_approx_kl", "approx_kl", "loss", "clipfrac", "lr"):
        out["upd_" + k] = np.array([u[k] for u in rec.updates])
    for k in ("mb_inds", "newlogprob", "entropy", "newvalue", "logits", "mb_advantages"):
        out["mb_" + k] = _stack(ups, k)
    for k in ("b_logprobs", "b_advantages", "b_returns", "b_values", "b_actions"):
        out[k] = ups[0][k]
    flat = lambda lst: np.concatenate([x.reshape(-1) for x in lst])
    out["grads_flat"] = np.stack([flat(u["grads"]) for u in ups])          # AFTER clip_grad_norm_
    out["params_before_flat"] = np.stack([flat(u["params_before"]) for u in ups])
    out["params_after_flat"] = np.stack([flat(u["params"]) for u in ups])
    out["param_shapes"] = np.array([list(x.shape) + [0] * (2 - x.ndim) for x in ups[0]["params"]])
    out["shuffles"] = np.stack(rec.shuffles)
    np.savez_compressed(OUT / name, **out)
    print("wrote", name)


def continuous(name, argv, n_iter):
    """cleanrl/ppo_continuous_action.py on the HalfCheetah-shaped synthetic env (obs 17, act 6)."""
    rec, g = run_reference("ppo_continuous_action.py", argv, gymnasium_kind="continuous")
    assert len(rec.iterations) == n_iter
    out = {"argv": np.array(argv)}
    for k in ("actions", "logprobs", "rewards", "dones", "values", "advantages", "returns", "next_value", "next_done",
              "param_sums"):
        out[k] = _stack(rec.iterations, k)
    for k in ("pg_loss", "v_loss", "entropy_loss", "old_approx_kl", "approx_kl", "loss", "clipfrac", "lr"):
        out["upd_" + k] = np.array([u[k] for u in rec.updates])
    out["upd_param_sums"] = _stack(rec.updates, "param_sums")
    out["shuffles"] = np.stack(rec.shuffles)
    out["state_dict_keys"] = np.array(list(g["agent"].state_dict().keys()))
    np.savez_compressed(OUT / name, **out)
    print("wrote", name)


def dqn(name, argv):
    """cleanrl/dqn_atari.py (+ the reference's own cleanrl_utils/buffers.py ReplayBuffer) on the synthetic
    gymnasium Atari env: every F.mse_loss value, the sampled index stream and the final parameters."""
    import torch
    import torch.nn.functional as F
    losses, qmeans, samples = [], [], []
    orig_mse = F.mse_loss

    def mse(a, b, *aa, **kk):
        out = orig_mse(a, b, *aa, **kk)
        losses.append(float(out.detach())); qmeans.append(float(b.detach().mean()))
        return out
    orig_randint = np.random.randint

    def randint(*a, **k):
        out = orig_randint(*a, **k)
        samples.append(np.array(out).reshape(-1)[:8].copy())
        return out
    F.mse_loss = mse
    np.random.randint = randint
    try:
        rec, g = run_reference("dqn_atari.py", argv, gymnasium_kind="atari")
    finally:
        F.mse_loss = orig_mse
        np.random.randint = orig_randint
    out = {"argv": np.array(argv), "td_losses": np.array(losses), "q_means": np.array(qmeans),
           "randint_heads": np.stack(samples[:64]) if samples else np.zeros((0, 8)),
           "param_sums": np.array([p.detach().double().sum().item() for p in g["q_network"].parameters()]),
           "param_abs_sums": np.array([p.detach().double().abs().sum().item() for p in g["q_network"].parameters()]),
           "state_dict_keys": np.array(list(g["q_network"].state_dict().keys()))}
    for t in sorted({t for t, _, _ in rec.scalars}):
        out["tb/" + t] = np.array([(s_, v) for tt, v, s_ in rec.scalars if tt == t], dtype=np.float64)
    np.savez_compressed(OUT / name, **out)
    print("wrote", name, len(losses), "updates")


SURFACE_SCRIPTS = ["ppo.py", "ppo_atari.py", "ppo_atari_envpool.py", "ppo_atari_multigpu.py", "ppo_continuous_action.py",
                   "dqn_atari.py", "ppo_procgen.py", "ppo_atari_lstm.py"]


def help_digest(text):
    """SHA-256 of a flag's help text (None when the flag has none): the fixture pins the text without holding it."""
    return None if text is None else hashlib.sha256(text.encode()).hexdigest()


def reference_surface(name):
    """The public surface of each reference script: every field of its ``Args`` dataclass as [name, default, help digest]
    (default "<expr>" where it is not a literal) and the names of its top-level classes and functions."""
    out = {}
    for script in SURFACE_SCRIPTS:
        tree = ast.parse((REFERENCE_ROOT / "cleanrl" / script).read_text())
        body = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "Args").body
        args = []
        for i, node in enumerate(body):
            if isinstance(node, ast.AnnAssign):
                try:
                    default = ast.literal_eval(node.value)
                except Exception:
                    default = "<expr>"
                doc = None
                if i + 1 < len(body) and isinstance(body[i + 1], ast.Expr) and isinstance(body[i + 1].value, ast.Constant):
                    doc = body[i + 1].value.value
                args.append([node.target.id, default, help_digest(doc)])
        out[script] = {"args": args,
                       "module_names": [n.name for n in tree.body if isinstance(n, (ast.ClassDef, ast.FunctionDef))]}
    (OUT / name).write_text(json.dumps(out, indent=1) + "\n")
    print("wrote", name)


def replay_buffer(name):
    """cleanrl_utils/buffers.py ReplayBuffer (optimize_memory_usage=True, 50 slots) fed 137 transitions of seeded random
    Atari frames, sampled 16 at a time (np.random.seed(t)) before and after the ring wraps.  Sampled frames are stored
    as the index of the generated frame they equal: the stream of frames is regenerated from the same seed."""
    from oracle import stubs
    from cleanrl_b200.synthetic_envs import Box, Discrete
    stubs.install()
    sys.path.insert(0, str(REFERENCE_ROOT))
    try:
        from cleanrl_utils.buffers import ReplayBuffer
        rng = np.random.default_rng(0)
        size, at = 50, (20, 49, 50, 77, 136)
        ref = ReplayBuffer(size, Box(0, 255, (4, 84, 84), np.uint8), Discrete(4), "cpu", optimize_memory_usage=True,
                           handle_timeout_termination=False)
        frames = [rng.integers(0, 256, (1, 4, 84, 84), dtype=np.uint8)]
        rec = {k: [] for k in ("observations", "next_observations", "actions", "rewards", "dones")}
        for t in range(137):
            frames.append(rng.integers(0, 256, (1, 4, 84, 84), dtype=np.uint8))
            a = rng.integers(0, 4, (1,)); r = rng.standard_normal(1).astype(np.float32); d = rng.random(1) < 0.1
            ref.add(frames[-2], frames[-1], a, r, d, [{}])
            if t in at:
                st = np.random.get_state()
                np.random.seed(t)
                data = ref.sample(16)
                np.random.set_state(st)
                for k in rec:
                    rec[k].append(getattr(data, k).numpy())
        index = {f.tobytes(): i for i, f in enumerate(frames)}
        out = {"sample_at": np.array(at)}
        for k in ("observations", "next_observations"):
            out[k + "_frame"] = np.array([[index[o.tobytes()] for o in x] for x in rec[k]])
        for k in ("actions", "rewards", "dones"):
            out[k] = np.stack([x.reshape(-1) for x in rec[k]])
    finally:
        sys.path.remove(str(REFERENCE_ROOT))
        stubs.uninstall()
    np.savez_compressed(OUT / name, **out)
    print("wrote", name, {k: (v.shape, v.dtype) for k, v in out.items()})


def main():
    OUT.mkdir(parents=True, exist_ok=True)
    only = sys.argv[1:]
    if not only or "ppo_atari_gym" in only:
        atari_envpool("ppo_atari_gym_n8_t32_seed2.npz",
                      ["--no-cuda", "--num-envs", "8", "--num-steps", "32", "--total-timesteps", "512", "--seed", "2"], 2,
                      script="ppo_atari.py")
    if not only or "ppo_atari_flags" in only:
        # flag coverage: no advantage normalisation, early stop on target_kl, other clip / coefficient values
        atari_envpool("ppo_atari_envpool_n8_t16_seed5_flags.npz",
                      ["--no-cuda", "--num-envs", "8", "--num-steps", "16", "--total-timesteps", "384", "--seed", "5",
                       "--no-norm-adv", "--target-kl", "0.0005", "--max-grad-norm", "0.3", "--vf-coef", "0.25",
                       "--clip-coef", "0.2", "--learning-rate", "1e-3"], 3)
    if not only or "ppo_atari_lstm" in only:
        atari_envpool("ppo_atari_lstm_n8_t16_seed4.npz",
                      ["--no-cuda", "--num-envs", "8", "--num-steps", "16", "--total-timesteps", "384", "--seed", "4"], 3,
                      script="ppo_atari_lstm.py", gymnasium_kind="atari1")
    if not only or "ppo_procgen" in only:
        atari_envpool("ppo_procgen_n8_t16_seed2.npz",
                      ["--no-cuda", "--num-envs", "8", "--num-steps", "16", "--total-timesteps", "384", "--seed", "2",
                       "--num-minibatches", "4", "--update-epochs", "2"], 3, script="ppo_procgen.py")
    if not only or "reference_surface" in only:
        reference_surface("reference_cli_surface.json")
    if not only or "replay_buffer" in only:
        replay_buffer("replay_buffer_n50_seed0.npz")
    if "ppo_atari_full" in only:
        # ~3 CPU-minutes: generated on request only (python -m oracle.make_golden ppo_atari_full)
        atari_envpool_full("ppo_atari_envpool_n1024_t128_seed1.npz",
                           ["--no-cuda", "--num-envs", "1024", "--num-steps", "128", "--total-timesteps", "131072", "--seed", "1"])
    if only:
        return
    dqn("dqn_atari_b8_seed1.npz",
        ["--no-cuda", "--total-timesteps", "260", "--learning-starts", "40", "--buffer-size", "64", "--batch-size", "8",
         "--train-frequency", "4", "--target-network-frequency", "20", "--seed", "1"])
    continuous("ppo_continuous_n4_t64_seed2.npz",
               ["--no-cuda", "--num-envs", "4", "--num-steps", "64", "--total-timesteps", "512", "--seed", "2",
                "--num-minibatches", "4", "--update-epochs", "2"], 2)
    atari_envpool("ppo_atari_envpool_n8_t32_seed1.npz",
                  ["--no-cuda", "--num-envs", "8", "--num-steps", "32", "--total-timesteps", "768", "--seed", "1"], 3)
    atari_envpool("ppo_atari_envpool_n16_t16_seed3_noclipv.npz",
                  ["--no-cuda", "--num-envs", "16", "--num-steps", "16", "--total-timesteps", "512", "--seed", "3",
                   "--no-clip-vloss", "--gamma", "0.98", "--gae-lambda", "0.9", "--no-anneal-lr",
                   "--update-epochs", "2", "--ent-coef", "0.02"], 2)
    mlp_ppo("ppo_mlp_n4_t128_seed1.npz",
            ["--no-cuda", "--num-envs", "4", "--num-steps", "128", "--total-timesteps", "1024", "--seed", "1"])


if __name__ == "__main__":
    sys.exit(main())
