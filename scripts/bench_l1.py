"""--distance 1 evaluation: the fused path (evaluate.evaluate_alignment_l1) against the materialised composition it
replaced (cdist -> csls_sim -> ranks on the [n, n] matrix) and, as context, the L2 fused evaluation on the same
inputs. One JSON line per workload on stdout. Timing: CUDA events, median over --steps after --warmup calls.

    python scripts/bench_l1.py --pairs 10500 --width 1200 --csls-k 10 [--steps 20 --warmup 3] [--no-materialised]
    torchrun --nproc-per-node 8 scripts/bench_l1.py --pairs 262144 --width 1200 --csls-k 10 --steps 3 --warmup 1 --no-materialised

Per kernel (one extra evaluation with every L1 sweep bracketed by events): ms, pairs/s and element-ops/s (pairs x D
over its time). Under torchrun every rank sweeps its shard of the targets; rank 0 prints, with a digest of the ranks
so that runs at different world sizes can be compared."""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from snag_b200 import evaluate, l1, ops  # noqa: E402


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = (q.stdout.splitlines()[0].split(", ") + ["?", "?", "?"])[:3] if q.returncode == 0 else ("?",) * 3
    return {"gpu": name, "power_limit": power, "sm_clock_max": clock}


def timed(fn, steps: int, warmup: int) -> tuple[float, object]:
    out = None
    for _ in range(warmup):
        out = fn()
    ts = []
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), out


class _KernelTimer:
    """Brackets the L1 sweep entry points of snag_b200.l1 with CUDA events for one evaluation."""

    def __init__(self):
        self.rec = []
        self.orig = {}

    def __enter__(self):
        for name, cols_arg in (("eval_rowtopk", 5), ("eval_rank", 11)):
            f = getattr(l1, name)
            self.orig[name] = f

            def wrap(*a, _f=f, _name=name, _c=cols_arg, **kw):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                r = _f(*a, **kw)
                e1.record()
                self.rec.append((_name, e0, e1, a[4] if _name == "eval_rowtopk" else a[10], a[_c], a[0].shape[1]))
                return r
            setattr(l1, name, wrap)
        return self

    def __exit__(self, *exc):
        for name, f in self.orig.items():
            setattr(l1, name, f)
        torch.cuda.synchronize()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=10500)
    ap.add_argument("--width", type=int, default=1200)
    ap.add_argument("--csls-k", type=int, default=10)
    ap.add_argument("--nocsls", action="store_true")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--no-materialised", action="store_true")
    ap.add_argument("--no-l2", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_l1.py measures on a GPU; none is visible")
    group, rank, world = None, 0, 1
    if "RANK" in os.environ:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist.init_process_group("nccl")
        group, rank, world = dist.group.WORLD, dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", torch.cuda.current_device())
    n, d, k, csls = a.pairs, a.width, a.csls_k, not a.nocsls
    gen = torch.Generator(device=dev).manual_seed(3408)
    x = torch.randn((n, d), device=dev, generator=gen)
    emb = torch.cat([x, x + 0.8 * torch.randn((n, d), device=dev, generator=gen)], 0)
    left, right = torch.arange(0, n, device=dev), torch.arange(n, 2 * n, device=dev)
    line = {"workload": f"l1_n{n}_d{d}_{'k%d' % k if csls else 'nocsls'}", "world": world, **gpu_info(),
            "steps": a.steps, "warmup": a.warmup}

    def fused():
        return evaluate.evaluate_alignment_l1(emb, left, right, csls=csls, csls_k=k, group=group)

    line["fused_ms"], out = timed(fused, a.steps, a.warmup)
    res = out["ranks"]
    line["deferred"] = l1.LAST_RANK_INFO.get("deferred")
    line["flagged_neighbourhoods"] = {t: v.get("flagged") for t, v in l1.LAST_TOPK_INFO.items()}
    line["ranks_digest"] = hashlib.sha256(res.rank_l2r.cpu().numpy().tobytes() + res.rank_r2l.cpu().numpy().tobytes()).hexdigest()[:16]
    line["mrr_l2r"] = out["l2r"].mrr
    with _KernelTimer() as kt:
        fused()
    kern = []
    for name, e0, e1, rows, cols, dp in kt.rec:
        ms = e0.elapsed_time(e1)
        kern.append({"kernel": name, "rows": rows, "cols": cols, "ms": round(ms, 3), "pairs_per_s": rows * cols / ms * 1e3,
                     "elem_ops_per_s": rows * cols * d / ms * 1e3})
    line["kernels"] = kern
    if world == 1 and not a.no_materialised:
        free, _ = torch.cuda.mem_get_info(dev)
        if 3 * 4 * n * n < free:
            def materialised():
                fe = torch.nn.functional.normalize(emb)
                dist = ops.l1_distance(fe[:n].contiguous(), fe[n:].contiguous())
                if csls:
                    o, _, _ = ops.csls_sim_matrix(1 - dist, k)
                    dist = 1 - o
                return ops.matrix_rank(dist)
            line["materialised_ms"], (r, c) = timed(materialised, a.steps, a.warmup)
            line["materialised_equal"] = bool(torch.equal(r, res.rank_l2r) and torch.equal(c, res.rank_r2l))
        else:
            line["materialised_ms"] = "does not fit"
    if not a.no_l2:
        line["l2_fused_ms"], _ = timed(lambda: evaluate.evaluate_alignment(emb, left, right, csls=csls, csls_k=k, group=group,
                                                                           graph=False), a.steps, a.warmup)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if group is not None:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
