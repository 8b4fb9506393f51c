"""CPU: the drop-in script's HOST logic against the committed reference fixtures.

tests/cpu_backend.py swaps the device kernels for the oracle / torch-CPU ops (in a subprocess, the product itself has
no CPU path), so what runs here is exactly the product's loop code: rollout bookkeeping, numpy shuffle consumption,
learning-rate annealing, --target-kl early stop, per-update statistics, TensorBoard tags and steps.  It must replay
the unmodified reference's runs recorded in tests/golden/ppo_atari_envpool_*.npz: same number of updates, same
losses, same scalars."""
import os
import subprocess
import sys
import textwrap
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden"

WORKER = textwrap.dedent('''
    import os, sys
    import numpy as np, torch
    sys.path.insert(0, ROOT); sys.path.insert(0, ROOT + "/tests")
    import cpu_backend
    cpu_backend.install()
    import importlib
    S = importlib.import_module("cleanrl_b200." + os.environ["SCRIPT"])
    z = np.load(os.environ["FIXTURE"])
    argv = [a for a in z["argv"].tolist()] + ["--synthetic-env"]
    class W:
        def __init__(self, *a): self.s = []
        def add_text(self, *a): pass
        def add_scalar(self, tag, v, step): self.s.append((tag, float(v), int(step)))
        def close(self): pass
    writers, snaps = [], []
    def wf(p):
        w = W(); writers.append(w); return w
    def on_it(it, eng, st):
        snaps.append({"actions": eng.actions.numpy().copy(), "advantages": eng.advantages.numpy().copy(),
                      "per_update": st["per_update"].copy()})
    S.main(argv, writer_factory=wf, on_iteration=on_it)
    tags = sorted({t for t, _, _ in writers[0].s})
    out = {"n_it": len(snaps), "actions": np.stack([s["actions"] for s in snaps]),
           "advantages": np.stack([s["advantages"] for s in snaps]),
           "per_update": np.concatenate([s["per_update"] for s in snaps]),
           "updates_per_it": np.array([s["per_update"].shape[0] for s in snaps])}
    for t in tags:
        out["tb/" + t] = np.array([(s, v) for tt, v, s in writers[0].s if tt == t], dtype=np.float64)
    np.savez(os.environ["OUT"], **out)
''')


@pytest.mark.parametrize("script,name", [
    ("ppo_atari_envpool", "ppo_atari_envpool_n8_t32_seed1.npz"),
    ("ppo_atari_envpool", "ppo_atari_envpool_n16_t16_seed3_noclipv.npz"),
    ("ppo_atari_envpool", "ppo_atari_envpool_n8_t16_seed5_flags.npz"),
    ("ppo_atari", "ppo_atari_gym_n8_t32_seed2.npz"),          # gymnasium-API loop (cleanrl/ppo_atari.py)
    ("ppo", "ppo_mlp_n4_t128_seed1.npz"),                     # MLP agent (cleanrl/ppo.py)
])
def test_host_loop_replays_reference_fixture(tmp_path, script, name):
    worker = tmp_path / "worker.py"
    worker.write_text(f"ROOT = {str(ROOT)!r}\n" + WORKER)
    out = tmp_path / "out.npz"
    # CUDA_VISIBLE_DEVICES="": the worker drives the CPU backend, so the script must take the CPU device on a GPU host too
    env = dict(os.environ, FIXTURE=str(GOLDEN / name), OUT=str(out), SCRIPT=script, OMP_NUM_THREADS="4", CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, str(worker)], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    z, o = np.load(GOLDEN / name), np.load(out)
    n_it = z["actions"].shape[0]
    assert int(o["n_it"]) == n_it
    # same number of minibatch updates (all epochs, or the reference's --target-kl early stops)
    assert o["per_update"].shape[0] == z["upd_loss"].shape[0], (o["updates_per_it"], z["upd_loss"].shape)
    # iteration 1 starts from identical weights and RNG streams: identical actions, advantages to fp32 rounding
    assert np.array_equal(o["actions"][0], z["actions"][0].astype(np.int64))
    assert np.abs(o["advantages"][0] - z["advantages"][0]).max() <= 1e-5 * max(1.0, np.abs(z["advantages"][0]).max())
    # per-update losses of iteration 1: right minibatches (numpy shuffle stream), right coefficients / flags
    k1 = int(o["updates_per_it"][0])
    for col, key in ((0, "upd_pg_loss"), (1, "upd_v_loss"), (2, "upd_entropy_loss"), (4, "upd_approx_kl"), (6, "upd_loss")):
        ref = z[key][:k1]
        tol = 1e-4 * np.maximum(1.0, np.abs(ref))
        assert (np.abs(o["per_update"][:k1, col] - ref) <= tol).all(), (key, o["per_update"][:k1, col], ref)
    # logged surface: same tags, same steps; learning rate exactly
    for key in z.files:
        if not key.startswith("tb/"):
            continue
        assert key in o.files, key
        if key.endswith("SPS") or "episodic" in key or "avg_" in key:
            continue
        assert np.array_equal(o[key][:, 0], z[key][:, 0]), key
    if "tb/charts/learning_rate" in z.files:
        assert np.array_equal(o["tb/charts/learning_rate"][:, 1], z["tb/charts/learning_rate"][:, 1])
