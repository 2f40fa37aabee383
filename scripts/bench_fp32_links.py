"""The trainer's link searches in fp32 (precision="fp32") against the default bf16 ones on the same inputs, at the sizes
the trainer runs them: one JSON line per size on stdout.

  mining  mining.iter_new_links(refresh=True) on n x n non-train rows (SNAG.Iter_new_links in the iterative-learning
          stage; DBP15K leaves ~15 500 non-train entities per side), D = 1200 (C1's joint width) and 1800;
  seeds   seeds.topk_similarity_entries at 15 000 x 15 000 image features, D = 2048 (DBP15K) and 4096 (FBDB15K),
          K = 100 * unsup_k (unsup_k = 1000, the reference's default), then the greedy matching of
          visual_pivot_induction.

    python scripts/bench_fp32_links.py [--steps 5 --warmup 1] > profiles/<name>.jsonl

Timing: CUDA events around the whole call (prologue included), median over --steps after --warmup calls. Inputs are
seeded on the device: clustered rows (64 centres), the right side a noisy permuted copy of the left (noise sigma: 8 for
mining, as in scripts/bench_fp32_eval.py, where about 87 % of the rows find their copy; 1 for the image features),
L2-normalised (image features additionally through a ReLU, as CNN features are non-negative). Per line: ms of each
mode, how many argmins (mining) or top-K entries (seeds) and how many links differ between the two modes, and the GPU's
name and power limit read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from bench_fp32_eval import gpu_info  # noqa: E402
from snag_b200 import mining, seeds  # noqa: E402


def clustered(n: int, d: int, sigma: float, seed: int, dev, relu: bool = False):
    g = torch.Generator(device=dev).manual_seed(seed)
    centres = torch.randn((64, d), generator=g, device=dev)
    x = torch.randn((n, d), generator=g, device=dev) + centres[torch.randint(0, 64, (n,), generator=g, device=dev)]
    y = (x + sigma * torch.randn((n, d), generator=g, device=dev))[torch.randperm(n, generator=g, device=dev)]
    if relu:
        x, y = x.clamp_min(0), y.clamp_min(0)
    return torch.nn.functional.normalize(x), torch.nn.functional.normalize(y)


def timed(fn, steps: int, warmup: int):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return out, round(float(np.median(ts)), 3)


def greedy(rows, cols, k: int):
    """visual_pivot_induction's one-to-one matching (src/data.py:381-394) on positions."""
    links, used_l, used_r = [], set(), set()
    for r, c in zip(rows.tolist(), cols.tolist()):
        if r in used_l or c in used_r:
            continue
        used_l.add(r)
        used_r.add(c)
        links.append((r, c))
        if len(links) == k:
            break
    return links


def bench_mining(n: int, d: int, sigma: float, steps: int, warmup: int, dev) -> dict:
    x, y = clustered(n, d, sigma, 3408, dev)
    emb = torch.cat([x, y], 0)
    del x, y
    left, right = list(range(n)), list(range(n, 2 * n))
    line = {"search": "mining", "n_left": n, "n_right": n, "width": d, "sigma": sigma}
    out = {}
    for prec in ("bf16", "fp32"):
        out[prec], line[f"ms_{prec}"] = timed(
            lambda: mining.iter_new_links(left, right, emb, [], True, precision=prec), steps, warmup)
    preds = {p: mining.mutual_nearest(emb[:n], emb[n:], precision=p) for p in ("bf16", "fp32")}
    line["argmins_differing"] = int((preds["bf16"][0] != preds["fp32"][0]).sum() + (preds["bf16"][1] != preds["fp32"][1]).sum())
    line["links_bf16"], line["links_fp32"] = len(out["bf16"]), len(out["fp32"])
    line["links_differing"] = len(set(out["bf16"]) ^ set(out["fp32"]))
    return line


def bench_seeds(n: int, d: int, sigma: float, unsup_k: int, steps: int, warmup: int, dev) -> dict:
    x, y = clustered(n, d, sigma, 3409, dev, relu=True)
    K = 100 * unsup_k
    line = {"search": "seeds", "n_left": n, "n_right": n, "width": d, "sigma": sigma, "K": K}
    out = {}
    for prec in ("bf16", "fp32"):
        out[prec], line[f"ms_{prec}"] = timed(
            lambda: seeds.topk_similarity_entries(x, y, K, precision=prec), steps, warmup)
    (rb, cb, _), (rf, cf, _) = out["bf16"], out["fp32"]
    line["topk_entries_differing"] = len(set(zip(rb.tolist(), cb.tolist())) ^ set(zip(rf.tolist(), cf.tolist())))
    line["topk_positions_differing"] = int(((rb != rf) | (cb != cf)).sum())
    lb, lf = greedy(rb.cpu(), cb.cpu(), unsup_k), greedy(rf.cpu(), cf.cpu(), unsup_k)
    line["seed_links_differing"] = len(set(lb) ^ set(lf))
    return line


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--mining-n", type=int, default=15500)
    ap.add_argument("--mining-widths", type=int, nargs="+", default=[1200, 1800])
    ap.add_argument("--mining-sigma", type=float, default=8.0)
    ap.add_argument("--seeds-n", type=int, default=15000)
    ap.add_argument("--seeds-widths", type=int, nargs="+", default=[2048, 4096])
    ap.add_argument("--seeds-sigma", type=float, default=1.0)
    ap.add_argument("--unsup-k", type=int, default=1000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    hw = gpu_info()
    for d in a.mining_widths:
        print(json.dumps({**bench_mining(a.mining_n, d, a.mining_sigma, a.steps, a.warmup, dev), **hw}), flush=True)
        torch.cuda.empty_cache()
    for d in a.seeds_widths:
        print(json.dumps({**bench_seeds(a.seeds_n, d, a.seeds_sigma, a.unsup_k, a.steps, a.warmup, dev), **hw}), flush=True)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
