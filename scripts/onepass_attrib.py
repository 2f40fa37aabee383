"""Attribution of the one-pass evaluation sweep (sim_kernel<EpiOnePass>): what its fp16x2 pre-filter flags, what the exact
fp32 tests make of the flagged elements, what is streamed, and the per-CTA cycle counters of the sweep. One JSON line per
configuration (stdout, and appended to --out).

    python scripts/onepass_attrib.py [--n 1000000,400000] [--gamma 1.5] [--sample 32768] [--out FILE]

Counts are whole-sweep totals over all CTAs:
  flagged_strips / flagged_cols / flagged_elems   warp strips (32 rows x 32 columns) with any flag, sum over those strips of
                                                  the flagged columns (union over the warp's rows), flagged elements
  accepted_row / accepted_col / accepted_l2r / accepted_r2l
                                                  flagged elements the exact test accepts: row top-k insertion, column
                                                  candidate appended, above the relaxed l2r / r2l rank threshold (an element
                                                  may count for several)
  accepted_none                                   flagged elements no exact test accepts: the price of the fp16 margin and of
                                                  testing the minimum of the thresholds
  streamed_rank / streamed_col                    entries appended to the rank and column-candidate streams
The cycle counters are per CTA (mean, and max over CTAs for the issuer wait): the UMMA issuer's total and its wait for a
free accumulator stage (> 0 means the epilogue held the tensor cores up), epilogue strip time and commit + barrier time.
The counters run in a separate, instrumented sweep (atomics on every flagged strip), so its time is not the product's;
ms_product is the same sweep without counters, timed with CUDA events in the same process.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import bench  # noqa: E402
from snag_b200 import _lib, evaluate, ops  # noqa: E402


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=10).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def run(n, gamma, sample, d=1200, k=10, sigma=6.0):
    dev = torch.device("cuda", 0)
    emb, left, right = bench.synth_tables(n, d, sigma, dev)
    X, xn = ops.prep_bf16(emb, left, True)
    Y, yn = ops.prep_bf16(emb, right, True)
    del emb
    sms = ops.num_sms()
    dbg = torch.zeros((4 * sms, 4), dtype=torch.int64, device=dev)
    evaluate.ONE_PASS_GAMMA = gamma
    evaluate.SAMPLE_MAX = sample
    orig = ops.eval_onepass
    rec = {}

    def wrapped(*a, **kw):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if rec.get("instrument"):
            dbg.zero_()
            _lib.call("snag_debug_counters", dbg.data_ptr())
        e0.record()
        out = orig(*a, **kw)
        e1.record()
        torch.cuda.synchronize()
        _lib.call("snag_debug_counters", None)
        rec["ms"] = e0.elapsed_time(e1)
        rec["stream_cnt"], rec["rk_cnt"] = out[4].clone(), out[7].clone()
        return out

    ops.eval_onepass = wrapped
    try:
        for _ in range(2):                                  # the second run finds the stream capacity the first one learnt
            rec["instrument"] = False
            evaluate.align_ranks(X, Y, xn, yn, n, k, True, one_pass=True)
        ms_product = rec["ms"]
        rec["instrument"] = True
        res = evaluate.align_ranks(X, Y, xn, yn, n, k, True, one_pass=True)
    finally:
        ops.eval_onepass = orig
    c = dbg.double().cpu()
    tot, wait, strip, tiles = (c[:sms, j].mean().item() for j in range(4))
    line = {
        "n": n, "d": d, "k": k, "gamma": gamma, "sample_max": sample, "gpu": gpu_info(),
        "ms_product": round(ms_product, 2), "ms_instrumented": round(rec["ms"], 2),
        "flagged_strips": int(c[sms:2 * sms, 1].sum()), "flagged_cols": int(c[sms:2 * sms, 2].sum()),
        "flagged_elems": int(c[sms:2 * sms, 3].sum()),
        "accepted_row": int(c[2 * sms:3 * sms, 0].sum()), "accepted_col": int(c[2 * sms:3 * sms, 1].sum()),
        "accepted_l2r": int(c[2 * sms:3 * sms, 2].sum()), "accepted_r2l": int(c[2 * sms:3 * sms, 3].sum()),
        "accepted_none": int(c[3 * sms:, 0].sum()),
        "streamed_rank": int(rec["rk_cnt"].long().sum()), "streamed_col": int(rec["stream_cnt"].long().sum()),
        "warp_strips": (n * n) // 1024,
        "issuer_clk_per_cta": round(tot), "issuer_wait_frac": round(wait / max(tot, 1), 4),
        "issuer_wait_max_frac": round(c[:sms, 1].max().item() / max(c[:sms, 0].max().item(), 1), 4),
        "tiles_per_cta": tiles, "epi_strip_clk_per_tile_per_warp": round(strip / 8 / max(tiles, 1)),
        "epi_commit_barrier_clk_per_tile_per_warp": round(c[sms:2 * sms, 0].mean().item() / 8 / max(tiles, 1)),
        "one_pass": res.info["one_pass"],
    }
    del X, Y, xn, yn
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", default="1000000,400000")
    ap.add_argument("--gamma", type=float, default=evaluate.ONE_PASS_GAMMA)
    ap.add_argument("--sample", type=int, default=evaluate.SAMPLE_MAX)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("onepass_attrib.py needs a GPU")
    for n in (int(v) for v in a.n.split(",")):
        line = json.dumps(run(n, a.gamma, a.sample))
        print(line, flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
