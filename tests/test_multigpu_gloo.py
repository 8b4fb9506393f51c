"""CPU, world_size = 2 over gloo: the data-parallel host path of cleanrl_b200/ppo_atari_multigpu.py
(reference: cleanrl/ppo_atari_multigpu.py:166-231,360-377; the reference's own test runs the script under
torchrun with gloo on CPU, tests/test_atari_multigpu.py:4-9).  Device kernels are replaced by the oracle
through tests/cpu_backend.py; what is under test is the product's host logic: per-rank seeding, env
sharding, ONE all-reduce of the flat gradient per update, /world_size folded into the optimiser step,
rank-0-only logging, global_step counting global envs."""
import os
import subprocess
import sys
import textwrap
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent

WORKER = textwrap.dedent('''
    import os, sys, json
    import numpy as np, torch, torch.distributed as dist
    sys.path.insert(0, ROOT); sys.path.insert(0, ROOT + "/tests")
    import cpu_backend
    cpu_backend.install()
    import importlib
    S = importlib.import_module("cleanrl_b200." + os.environ["SCRIPT"])
    rank = int(os.environ["LOCAL_RANK"])
    calls = {"n": 0, "numel": []}
    orig = dist.all_reduce
    def counting(t, op=dist.ReduceOp.SUM, **k):
        calls["n"] += 1; calls["numel"].append(t.numel())
        return orig(t, op=op, **k)
    dist.all_reduce = counting
    class W:
        def __init__(self, *a): self.s = []
        def add_text(self, *a): pass
        def add_scalar(self, tag, v, step): self.s.append((tag, float(v), int(step)))
        def close(self): pass
    writers = []
    def wf(p):
        w = W(); writers.append(w); return w
    snaps = []
    def on_it(it, eng, st):
        snaps.append({"actions": eng.actions.numpy().copy(), "flat": eng.flat.flat.numpy().copy(), "st": st["per_update"].copy()})
    extra = ["--backend", "gloo"] if os.environ["SCRIPT"].endswith("envpool") else []
    eng = S.main(["--local-num-envs", "4", "--num-steps", "8", "--total-timesteps", "128", "--update-epochs", "2",
                  "--no-cuda", "--synthetic-env", "--seed", "5"] + extra, writer_factory=wf, on_iteration=on_it)
    if os.environ["SCRIPT"].endswith("envpool"):
        # per-rank core pinning: disjoint, equal slices of the cores this job may use
        import json
        mine = sorted(os.sched_getaffinity(0))
        with open(os.environ["OUT"] + f"/cores{rank}.json", "w") as f:
            json.dump({"mine": mine, "engine": list(eng.env_cores)}, f)
    np.savez(os.environ["OUT"] + f"/rank{rank}.npz", flat=np.stack([s["flat"] for s in snaps]),
             actions=np.stack([s["actions"] for s in snaps]), n_allreduce=calls["n"], numel=np.array(calls["numel"]),
             n_writers=len(writers), tags=np.array(sorted({t for w in writers for t, _, _ in w.s})),
             steps=np.array(sorted({s for w in writers for _, _, s in w.s})), P=eng.flat.numel)
    dist.destroy_process_group()
''')


@pytest.mark.parametrize("module", ["ppo_atari_multigpu", "ppo_atari_multigpu_envpool"])
def test_two_rank_gloo_data_parallel(tmp_path, module):
    script = tmp_path / "worker.py"
    script.write_text(f"ROOT = {str(ROOT)!r}\n" + WORKER)
    # CUDA_VISIBLE_DEVICES="": the ranks drive the CPU backend, so the script must take the CPU device on a GPU host too
    env = dict(os.environ, OUT=str(tmp_path), OMP_NUM_THREADS="2", SCRIPT=module, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nnodes=1", "--nproc-per-node=2",
                        "--local-addr", "127.0.0.1", str(script)], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    z0, z1 = np.load(tmp_path / "rank0.npz"), np.load(tmp_path / "rank1.npz")
    # replicas stay bit-identical after every iteration (same init via seed - rank, same averaged gradient)
    assert np.array_equal(z0["flat"], z1["flat"])
    # different env / sampling streams per rank
    assert not np.array_equal(z0["actions"], z1["actions"])
    # ONE all-reduce of the whole flat gradient per minibatch update: 2 iterations x 2 epochs x 4 minibatches
    assert int(z0["n_allreduce"]) == 16 and int(z1["n_allreduce"]) == 16
    assert set(z0["numel"].tolist()) == {int(z0["P"]) + (-int(z0["P"])) % 4}
    # rank-0-only writer; global_step counts GLOBAL envs: 8 envs x 8 steps per iteration
    assert int(z0["n_writers"]) == 1 and int(z1["n_writers"]) == 0
    assert {"charts/SPS", "losses/value_loss", "losses/clipfrac", "charts/learning_rate"} <= set(z0["tags"].tolist())
    assert 64 in z0["steps"].tolist() and 128 in z0["steps"].tolist()
    assert "local_rank: 1" in r.stdout and "agent.actor.weight.sum()" in r.stdout
    if module.endswith("envpool"):
        import json
        c0, c1 = (json.loads((tmp_path / f"cores{k}.json").read_text()) for k in (0, 1))
        assert c0["mine"] == c0["engine"] and c1["mine"] == c1["engine"]
        assert not set(c0["mine"]) & set(c1["mine"]) and len(c0["mine"]) == len(c1["mine"]) >= 1


def test_world1_matches_averaged_two_rank_gradient_math():
    """clip_adam(world_size=2) on the SUM of two gradients == clip_adam(world_size=1) on their mean
    (the identity the fused /world_size relies on), via the oracle."""
    from oracle import ppo_oracle as O
    rng = np.random.default_rng(0)
    p = rng.standard_normal(1000).astype(np.float32); m = np.zeros(1000, np.float32); v = np.zeros(1000, np.float32)
    g0, g1 = rng.standard_normal(1000).astype(np.float32), rng.standard_normal(1000).astype(np.float32)
    a = O.clip_adam(p, g0 + g1, m, v, 1, 1e-3, world_size=2)
    b = O.clip_adam(p, (g0 + g1) / np.float32(2), m, v, 1, 1e-3, world_size=1)
    assert np.array_equal(a[0], b[0])


def test_core_slices_partition_the_host():
    """ppo_atari_multigpu_envpool.core_slice: ranks get disjoint, equal, contiguous shares of the allowed cores
    (docs/rl-algorithms/ppo.md:1020: pin the env threads of each subprocess so the pools do not fight)."""
    from cleanrl_b200.ppo_atari_multigpu_envpool import core_slice
    cores = list(range(3, 67))                    # 64 allowed cores, not starting at 0
    parts = [core_slice(r, 8, cores) for r in range(8)]
    assert all(len(p) == 8 for p in parts)
    assert sorted(c for p in parts for c in p) == cores
    assert all(p == list(range(p[0], p[0] + 8)) for p in parts)
    assert core_slice(0, 1, cores) == cores
    assert len(core_slice(5, 8, [0, 1])) == 1    # more ranks than cores: still one core each
