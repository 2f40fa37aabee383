"""The fp32 evaluation (evaluate_alignment(precision="fp32")) against the default bf16 one on the same inputs: one JSON
line per size and mode on stdout. Timing: CUDA events around the whole call (prologue included), median over --steps
after --warmup calls. Inputs: 2n clustered rows (64 centres, targets = noisy copies of the sources), D = --width,
seeded on the device.

    python scripts/bench_fp32_eval.py --pairs 10500 100000 1000000 --width 1200 --csls-k 10 [--steps 5 --warmup 1]

Per line: median ms, the sweeps executed (kernel names, from one extra evaluation with every sweep bracketed by events),
the elements deferred to the canonical re-score, the neighbourhoods flagged for verification (rows / cols) and, on the
fp32 line, how many ranks and whether Hits@1 / MRR differ from the bf16 mode."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from snag_b200 import evaluate, ops  # noqa: E402


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = (q.stdout.splitlines()[0].split(", ") + ["?", "?", "?"])[:3] if q.returncode == 0 else ("?",) * 3
    return {"gpu": name, "power_limit": power, "sm_clock_max": clock}


def problem(n: int, d: int, sigma: float, seed: int, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    centres = torch.randn((64, d), generator=g, device=dev)
    x = torch.randn((n, d), generator=g, device=dev) + centres[torch.randint(0, 64, (n,), generator=g, device=dev)]
    y = x + sigma * torch.randn((n, d), generator=g, device=dev)
    emb = torch.cat([x, y], 0)
    del x, y
    ar = torch.arange(n, device=dev)
    return emb, ar, ar + n


def counts(res) -> dict:
    info = res.info
    nb = info.get("neighbourhoods", {})
    one = info.get("one_pass")
    deferred = one["deferred"] if one and one.get("fallback") is None else info.get("rank_sweep", {}).get("deferred")
    return {"deferred": deferred, "flagged_rows": nb.get("rows", {}).get("flagged"),
            "flagged_cols": nb.get("cols", {}).get("flagged"), "one_pass": one is not None and one.get("fallback") is None}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, nargs="+", default=[10500, 100000, 1000000])
    ap.add_argument("--width", type=int, default=1200)
    ap.add_argument("--csls-k", type=int, default=10)
    ap.add_argument("--sigma", type=float, default=8.0)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    hw = gpu_info()
    for n in a.pairs:
        emb, left, right = problem(n, a.width, a.sigma, 3408, dev)
        out = {}
        for prec in ("bf16", "fp32"):
            def run():
                return evaluate.evaluate_alignment(emb, left, right, True, a.csls_k, graph=False, precision=prec)
            for _ in range(a.warmup):
                run()
            ts = []
            for _ in range(a.steps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                r = run()
                e1.record()
                e1.synchronize()
                ts.append(e0.elapsed_time(e1))
            sweeps = []
            ops.SWEEP_EVENT_SINK = sweeps
            try:
                run()
            finally:
                ops.SWEEP_EVENT_SINK = None
            torch.cuda.synchronize()
            out[prec] = r
            line = {"pairs": n, "width": a.width, "csls_k": a.csls_k, "precision": prec, "ms": round(float(np.median(ts)), 3),
                    "sweeps": [(nm, round(e0.elapsed_time(e1), 3)) for nm, e0, e1, *_ in sweeps], **counts(r["ranks"]),
                    "hits1_l2r": float(r["l2r"].acc[0]), "mrr_l2r": r["l2r"].mrr, "mrr_r2l": r["r2l"].mrr,
                    "peak_mem_gb": round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 2), **hw}
            if prec == "fp32":
                b, f = out["bf16"], out["fp32"]
                line["ranks_differing"] = int((b["ranks"].rank_l2r != f["ranks"].rank_l2r).sum() +
                                              (b["ranks"].rank_r2l != f["ranks"].rank_r2l).sum())
                line["hits1_differs"] = bool(b["l2r"].acc[0] != f["l2r"].acc[0] or b["r2l"].acc[0] != f["r2l"].acc[0])
                line["mrr_differs"] = bool(b["l2r"].mrr != f["l2r"].mrr or b["r2l"].mrr != f["r2l"].mrr)
            print(json.dumps(line), flush=True)
            torch.cuda.reset_peak_memory_stats(dev)
        del emb, left, right, out
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
