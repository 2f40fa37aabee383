"""The command-line contract of bench.py. Without a GPU: the reference arm (the CPU port of the path timed on the host cores)
prints exactly ONE line on stdout, a JSON object carrying the result keys; under torchrun only rank 0 prints; arguments it
cannot honour are refused. On the GPU: --dump-outputs writes what the timed path computed."""
from __future__ import annotations

import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CONTRACT_KEYS = ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                 "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches")


def _run(cmd, env=None):
    r = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return [ln for ln in r.stdout.splitlines() if ln.strip()]


def _check_line(line: dict, n_gpus: int):
    for key in CONTRACT_KEYS:
        assert key in line, key
    assert line["impl"] == "reference" and line["n_gpus"] == n_gpus and line["gpu_launches"] == 0
    assert line["metric"].startswith("align-eval entity pairs/sec") and line["unit"] == "pairs/s"
    assert line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["config"]["workload"] == "c4_1m" and "model" not in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sub-problem" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["value"] > 0 and line["ms_per_step"] > 0


def test_reference_arm_prints_one_json_line():
    out = _run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0"])
    assert len(out) == 1, out
    _check_line(json.loads(out[0]), 1)


def test_reference_arm_under_torchrun_only_rank0_prints():
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                "--master-port", "29533", "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], env)
    lines = [ln for ln in out if ln.startswith("{")]
    assert len(lines) == 1, out
    _check_line(json.loads(lines[0]), 2)


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_refuses_bad_arguments(argv, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], cwd=tmp_path, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=120)
    assert r.returncode == 2 and "error:" in r.stderr and r.stdout == ""
    assert not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_dump_outputs_equal_the_timed_path(cuda_device, tmp_path):
    """--dump-outputs writes what the timed path computed in its last step, from inputs that are the same in every run:
    the evaluation's outputs equal a fresh in-process evaluation of bench.synth_tables bit for bit, and the training
    slice's loss and sampled gradients equal one eager step on bench._train_tables."""
    import numpy as np
    import torch
    import bench
    from snag_b200 import evaluate, loss as sloss, ops
    for workload in ("c1", "c1_train"):
        out = _run([sys.executable, "bench.py", "--workload", workload, "--steps", "2", "--warmup", "0", "--no-train",
                    "--no-audit", "--no-context", "--dump-outputs", str(tmp_path)])
        assert json.loads(out[-1])["steps"] == 2
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())

    n, d, k, sigma, _ = bench.WORKLOADS["c1"]
    emb, left, right = bench.synth_tables(n, d, sigma, cuda_device)
    X, xn = ops.prep_bf16(emb, left, True)
    Y, yn = ops.prep_bf16(emb, right, True)
    res = evaluate.align_ranks(X, Y, xn, yn, n, k, True, False)
    for nm in ("rank_l2r", "rank_r2l", "nv1", "nv2", "g"):
        np.testing.assert_array_equal(got[f"c1.{nm}"], getattr(res, nm).cpu().numpy(), err_msg=nm)
    assert got["c1.rank_l2r"].dtype == np.float64 and got["c1.nv1"].dtype == np.float32

    B, M, dm, _ = bench.TRAIN_WORKLOADS["c1_train"]
    streams, hidden, joint, joint_fz, wn, links, _leaves = bench._train_tables(B, M, dm, cuda_device)
    layer = sloss.SnagLossLayer(tau=0.1, ab_weight=0.5).to(cuda_device)
    lv = layer(streams, hidden, joint, joint_fz, torch.from_numpy(links).to(cuda_device), wn)
    lv.backward()
    np.testing.assert_allclose(got["c1_train.loss"], [lv.item()], rtol=1e-5)
    rows = np.sort(np.random.RandomState(bench.SEED + 2).choice(wn.shape[0], bench.DUMP_ROWS, replace=False))
    named = [(f"stream{m}", t) for m, t in enumerate(streams)] + [(f"hidden{m}", t) for m, t in enumerate(hidden)]
    named += [("joint", joint), ("joint_fz", joint_fz), ("weight_norm", wn)]
    named = [(nm, t) for nm, t in named if t is not None]
    assert sorted(f"c1_train.grad_{nm}" for nm, _ in named) == sorted(g for g in got if g.startswith("c1_train.grad_"))
    for nm, t in named:
        want = t.grad[torch.from_numpy(rows).to(cuda_device)].cpu().numpy()
        a = got[f"c1_train.grad_{nm}"]
        assert a.shape == want.shape and np.linalg.norm(a - want) <= 1e-4 * np.linalg.norm(want), nm
