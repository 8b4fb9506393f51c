"""CPU tests: the C-ABI library builds for sm_100a, loads, and exports every symbol
include/b200rl.h declares; the CLI surface matches the reference; the product has no
CPU fallback and never imports the oracle."""
import ctypes
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def _declared_symbols():
    txt = (ROOT / "include" / "b200rl.h").read_text()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(b200rl_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol(lib):
    syms = _declared_symbols()
    assert len(syms) >= 15
    raw = ctypes.CDLL(str(ROOT / "cleanrl_b200" / "libb200rl.so"))
    for s in syms:
        assert hasattr(raw, s), f"{s} declared in include/b200rl.h but not exported"
    from cleanrl_b200 import _lib
    assert sorted(_lib.SIGNATURES) == syms, "python binding table out of sync with the header"
    assert lib.b200rl_compiled_arch() == 100
    assert lib.b200rl_version() >= 100


def test_library_contains_sm100a_code_only():
    out = subprocess.run(["cuobjdump", "-lelf", str(ROOT / "cleanrl_b200" / "libb200rl.so")], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    archs = set(re.findall(r"sm_(\d+a?)", out.stdout))
    assert archs == {"100a"}, archs


def test_argument_validation_without_gpu(lib):
    """Validation happens before any CUDA call, so it is testable on a CPU-only box."""
    rc = lib.b200rl_gae_f32(None, None, None, None, None, None, None, 4, 4, 0.99, 0.95, 0, None)
    assert rc == -1 and b"null" in lib.b200rl_last_error()
    rc = lib.b200rl_gae_f32(None, None, None, None, None, None, None, 0, 4, 0.99, 0.95, 0, None)
    assert rc == 0  # empty rollout is a no-op
    rc = lib.b200rl_categorical_sample_f32(1, 4, 1, None, 0, 8, 100, 1, 1, None, None, None)
    assert rc == -1 and b"outside" in lib.b200rl_last_error()
    rc = lib.b200rl_clip_adam_f32(16, 16, 16, 16, 8, 0, 1e-3, 0.9, 0.999, 1e-5, 0.5, 1, None, 16, 1 << 20, None)
    assert rc == -1 and b"1-based" in lib.b200rl_last_error()
    rc = lib.b200rl_ppo_loss_f32(16, 4, 16, 1, None, 16, 16, 16, 16, 16, 8, 4, .1, .01, .5, 1, 1, 16, 4, 16, 1, 16, 16, 8, None)
    assert rc == -4  # workspace too small


def test_ops_reject_cpu_tensors(lib):
    import torch
    from cleanrl_b200 import ops
    x = torch.zeros(4, 4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.gae(x, x, x, x[0], x[0], 0.99, 0.95)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.clip_adam(x.view(-1), x.view(-1), x.view(-1), x.view(-1), 1, 1e-3)


def test_script_refuses_to_run_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from cleanrl_b200 import ppo_atari_envpool as S

    class W:
        def __init__(self, *a): pass
        def add_text(self, *a): pass
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        S.main(["--num-envs", "2", "--num-steps", "4", "--total-timesteps", "8"], writer_factory=W)


def test_product_never_imports_oracle():
    for p in list((ROOT / "cleanrl_b200").rglob("*.py")):
        txt = p.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f"{p} imports the oracle"


def _reference_surface(script):
    """Args fields and top-level names of the reference script, recorded in tests/golden/reference_cli_surface.json
    (oracle/make_golden.py reference_surface)."""
    import json
    return json.loads((ROOT / "tests" / "golden" / "reference_cli_surface.json").read_text())[script]


@pytest.mark.parametrize("script,factory", [
    ("ppo.py", "ppo_args"), ("ppo_atari.py", "ppo_atari_args"), ("ppo_atari_envpool.py", "ppo_atari_envpool_args"),
    ("ppo_atari_multigpu.py", "ppo_atari_multigpu_args"), ("ppo_continuous_action.py", "ppo_continuous_action_args"),
    ("dqn_atari.py", "dqn_atari_args"), ("ppo_procgen.py", "ppo_procgen_args"),
    ("ppo_atari_lstm.py", "ppo_atari_args")])
def test_cli_fields_match_reference_args(script, factory):
    """Every reference flag exists with the same default and help text (reference Args dataclasses)."""
    import dataclasses
    from cleanrl_b200 import cli
    from oracle.make_golden import help_digest
    ref = {name: (default, digest) for name, default, digest in _reference_surface(script)["args"]}
    assert ref
    ours = getattr(cli, factory)()
    fields = {f.name: f for f in dataclasses.fields(ours)}
    for name, (default, digest) in ref.items():
        assert name in fields, f"{script}: flag {name} missing"
        f = fields[name]
        if default != "<expr>":
            d = f.default if f.default is not dataclasses.MISSING else f.default_factory()
            assert d == default, (name, d, default)
        helps = [m.help for m in getattr(f.type, "__metadata__", ()) if hasattr(m, "help")]
        assert helps and help_digest(helps[0]) == digest, (name, helps)
    extra = set(fields) - set(ref)
    assert extra <= {"precision", "gae_kernel", "synthetic_env", "huber_loss", "env_groups"}, extra


@pytest.mark.parametrize("script", ["ppo.py", "ppo_atari.py", "ppo_atari_envpool.py", "ppo_atari_multigpu.py",
                                    "ppo_continuous_action.py", "dqn_atari.py"])
def test_module_level_names_match_reference(script):
    """Every top-level class / function of the reference script (what tuner.py, the eval helpers and user code
    import: Args, make_env, layer_init, Agent / QNetwork, RecordEpisodeStatistics, linear_schedule) exists in the
    drop-in module under the same name."""
    import importlib
    names = _reference_surface(script)["module_names"]
    mod = importlib.import_module("cleanrl_b200." + script[:-3])
    missing = [n for n in names if not hasattr(mod, n)]
    assert names and not missing, (script, missing)


def test_cartpole_vec_dynamics_and_episode_bookkeeping():
    """CartPoleVec (host-side env for the learning-curve test): a random policy lasts ~22 steps on average, a
    bang-bang controller on the pole angle + angular velocity reaches the 500-step truncation, and final_info
    carries return == length at every episode end."""
    from cleanrl_b200.synthetic_envs import CartPoleVec
    env = CartPoleVec(4)
    obs, _ = env.reset(seed=1)
    rng = np.random.default_rng(0)
    rets = []
    for _ in range(4000):
        obs, r, te, tr, info = env.step(rng.integers(0, 2, 4))
        assert obs.dtype == np.float32 and obs.shape == (4, 4) and (r == 1).all() and not (te & tr).any()
        if "final_info" in info:
            for i, f in enumerate(info["final_info"]):
                assert (f is not None) == bool(te[i] or tr[i])
                if f is not None:
                    assert float(f["episode"]["r"][0]) == float(f["episode"]["l"][0])
                    rets.append(float(f["episode"]["r"][0]))
    assert 15 < np.mean(rets) < 35, np.mean(rets)
    obs, _ = env.reset(seed=2)
    truncs = 0
    for _ in range(1200):
        obs, r, te, tr, info = env.step((obs[:, 2] + 0.5 * obs[:, 3] > 0).astype(np.int64))
        truncs += int(tr.sum())
        if "final_info" in info:
            for f in info["final_info"]:
                if f is not None:
                    assert float(f["episode"]["r"][0]) <= 500
    assert truncs >= 4, truncs


def test_native_minibatch_shuffle_is_numpy_shuffle_bit_for_bit(lib):
    """b200rl_mt19937_shuffle_i64 == np.random.shuffle on the global RandomState (the reference's minibatch shuffle,
    cleanrl/ppo.py:245): same permutations, and the generator is left in the same state (later draws agree)."""
    from cleanrl_b200 import ops
    for seed in (0, 1, 7, 2 ** 31 - 1):
        for n in (1, 2, 3, 17, 1000, 4 * 128, 131072):
            np.random.seed(seed)
            np.random.random(seed % 5)                    # generator position anywhere inside the 624-word block
            a = np.arange(n)
            for _ in range(3):                            # cumulative, in place, as the epochs of an update
                np.random.shuffle(a)
            tail_a = np.random.randint(0, 1 << 30, size=5)
            np.random.seed(seed)
            np.random.random(seed % 5)
            b = np.arange(n)
            for _ in range(3):
                ops.numpy_global_shuffle(b)
            tail_b = np.random.randint(0, 1 << 30, size=5)
            assert np.array_equal(a, b) and np.array_equal(tail_a, tail_b), (seed, n)
    # anything that is not a contiguous int64 vector takes numpy's own path
    np.random.seed(3); x = np.arange(10, dtype=np.int32); np.random.shuffle(x)
    np.random.seed(3); y = np.arange(10, dtype=np.int32); ops.numpy_global_shuffle(y)
    assert np.array_equal(x, y)


def test_frame_stack_entry_points_validate_arguments_without_gpu(lib):
    """The round-2 entry points (frame-stack delta upload, device-scalar Adam, native shuffle) reject bad arguments before
    touching CUDA; ops.* reject CPU tensors."""
    import torch
    from cleanrl_b200 import ops
    assert lib.b200rl_frames_delta_s2d_u8(None, None, None, None, None, 4, None, None, None) == -1
    assert b"null" in lib.b200rl_last_error()
    assert lib.b200rl_frames_delta_s2d_u8(None, None, None, None, None, 0, None, None, None) == 0      # empty batch: no-op
    assert lib.b200rl_frames_delta_s2d_u8(16, 16, None, 32, 48, 4, 64, 80, None) == -1                # slot table without frames
    assert lib.b200rl_frames_delta_s2d_u8(16, None, None, 32, 48, 4, 32, 80, None) == -1              # in place
    assert b"in-place" in lib.b200rl_last_error()
    assert lib.b200rl_h2d_rows_async(16, 16, 8, 16, 4, None) == -1                                    # pitch < row
    assert lib.b200rl_h2d_rows_async(None, None, 16, 16, 0, None) == 0
    assert not lib.b200rl_stackdelta_create(0, 4, 7056, 2) and b"stackdelta_create" in lib.b200rl_last_error()
    assert not lib.b200rl_stackdelta_create(8, 1, 7056, 2)
    tr = ops.StackDeltaTracker(4, 4, 64, threads=1, pinned=False)
    obs = np.zeros((4, 4, 8, 8), dtype=np.uint8)
    assert lib.b200rl_stackdelta_begin(tr._h, obs.ctypes.data, 8, None, None, tr.full_h.data_ptr(), tr.slot_h.data_ptr()) == -1
    assert b"env_stride" in lib.b200rl_last_error()
    assert lib.b200rl_stackdelta_begin(None, None, 0, None, None, None, None) == -1
    assert lib.b200rl_stackdelta_wait(None, None) == -1
    assert lib.b200rl_stackdelta_join(None, None, None) == 0                                          # nothing pending
    assert lib.b200rl_stackdelta_launch(None, None, 0, None) == -1
    assert lib.b200rl_clip_adam_dyn_f32(16, 16, 16, 16, 8, None, 0.9, 0.999, 1e-5, 0.5, 1, None, 16, 1 << 20, None) == -1
    assert b"scalar table" in lib.b200rl_last_error()
    import ctypes
    out = (ctypes.c_float * 2)()
    assert lib.b200rl_adam_step_scalars(0, 1e-3, 0.9, 0.999, out) == -1 and lib.b200rl_adam_step_scalars(1, 1e-3, 0.9, 0.999, out) == 0
    assert abs(out[0] - (1 - 0.999) ** 0.5) < 1e-7 and abs(out[1] + 1e-3 / (1 - 0.9)) < 1e-9
    key = np.zeros(624, dtype=np.uint32)
    pos = ctypes.c_int32(700)
    assert lib.b200rl_mt19937_shuffle_i64(key.ctypes.data, ctypes.addressof(pos), None, 0) == -1      # position outside the block
    x = torch.zeros(4, 7056, dtype=torch.uint8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.frames_delta_s2d_u8(x, x, x, x, x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.clip_adam_dyn(torch.zeros(8), torch.zeros(8), torch.zeros(8), torch.zeros(8), torch.zeros(2))


def test_public_header_is_plain_c(tmp_path):
    """include/b200rl.h is the drop-in boundary: it must compile as C99 (no C++, no torch / CUDA types in the signatures)."""
    import shutil
    if shutil.which("gcc") is None:
        pytest.skip("gcc unavailable")
    src = tmp_path / "hdr.c"
    src.write_text('#include "b200rl.h"\nint main(void) { B200rlPartLaunch p; (void)p; return b200rl_version() ? 0 : 1; }\n')
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-I", str(ROOT / "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    txt = (ROOT / "include" / "b200rl.h").read_text()
    assert "#include <cuda" not in txt and "at::" not in txt and "std::" not in txt
