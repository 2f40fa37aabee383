"""Dev probe: where the time of the fused evaluation sweeps goes (per-CTA cycle counters of sim_kernel): UMMA issuer total,
its wait for a free accumulator stage (= the epilogue is the bottleneck), epilogue strip time, barrier time."""
import json
import sys

import torch

sys.path.insert(0, ".")
import bench  # noqa: E402
from snag_b200 import _lib, evaluate, ops  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 400_000
gamma = float(sys.argv[2]) if len(sys.argv) > 2 else 1.5
d, k, sigma = 1200, 10, 6.5
dev = torch.device("cuda", 0)
emb, left, right = bench.synth_tables(n, d, sigma, dev)
X, xn = ops.prep_bf16(emb, left, True)
Y, yn = ops.prep_bf16(emb, right, True)
del emb
sms = ops.num_sms()
dbg = torch.zeros((4 * sms, 4), dtype=torch.int64, device=dev)   # rows 2*sms.. : EpiOnePass per-test counters
records = []


def smi():
    import subprocess
    try:
        o = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,power.draw,clocks_event_reasons.active", "--format=csv,noheader,nounits",
                            "-i", "0"], capture_output=True, text=True, timeout=5).stdout.strip()
        return o
    except Exception as e:  # noqa: BLE001
        return str(e)



def wrap(name):
    fn = getattr(ops, name)

    def w(*a, **kw):
        dbg.zero_()
        torch.cuda.synchronize()
        _lib.call("snag_debug_counters", dbg.data_ptr())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn(*a, **kw)
        e1.record()
        import time as _t
        _t.sleep(0.12)
        during = smi()
        torch.cuda.synchronize()
        _lib.call("snag_debug_counters", None)
        c = dbg.double().cpu()
        ms = e0.elapsed_time(e1)
        tot, wait, strip, tiles = c[:sms, 0].mean().item(), c[:sms, 1].mean().item(), c[:sms, 2].mean().item(), c[:sms, 3].mean().item()
        bar = c[sms:, 0].mean().item()
        fl = [c[sms:, j].sum().item() for j in (1, 2, 3)]
        tmin, tmax = c[:sms, 0].min().item(), c[:sms, 0].max().item()
        wmax = c[:sms, 1].max().item()
        records.append({"flag_strips_cols_elems_per_warpstrip": [round(v / (n * n / 1024.0), 3) for v in fl], "kernel": name, "ms": round(ms, 2), "sm_mhz": round(tot / ms / 1e3, 0), "sm_mhz_from_max": round(tmax / ms / 1e3, 0),
                        "issuer_clk_min_max": [tmin, tmax], "issuer_wait_max_frac": round(wmax / tmax, 3), "smi_during": during, "tiles_per_cta": tiles,
                        "clk_per_tile": round(tot / max(tiles, 1)), "issuer_wait_frac": round(wait / tot, 3),
                        "epi_strip_clk_per_tile_per_warp": round(strip / 8 / max(tiles, 1)),
                        "epi_commit_barrier_clk_per_tile_per_warp": round(bar / 8 / max(tiles, 1))})
        return out
    setattr(ops, name, w)


for nm in ("eval_rowcoltopk", "eval_onepass", "eval_rank"):
    wrap(nm)
evaluate.ONE_PASS_GAMMA = gamma
for one in (False, True, False, True):
    records.clear()
    res = evaluate.align_ranks(X, Y, xn, yn, n, k, True, one_pass=one)
    for r in records:
        print(json.dumps(r), flush=True)
    if one:
        print(json.dumps(res.info["one_pass"]), flush=True)
