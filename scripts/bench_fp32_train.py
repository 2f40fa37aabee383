"""The loss-layer slice of a training step (SnagLossLayer: 2 + 2M icl_loss calls, forward + backward) with the fp32
training route (precision="fp32", snag_b200.loss_fp32) against the default bf16 route, on the inputs of bench.py's
c1_train and c5_train workloads, one GPU: one JSON line per (workload, precision) and one line per checked table.

    python scripts/bench_fp32_train.py [--steps 10 --warmup 3] [--out profiles/r11_fp32_train_bench_n1.jsonl]

Timing: CUDA events around each eager step (zeroed gradients, forward, backward), median over --steps after --warmup
steps. Errors: per precision, the largest per-anchor NLL error and the largest d emb row error (relative to the largest
row) of one icl_loss call on a table of the timed inputs, against the fp64 loss of the unrounded normalised fp32 rows
(tests/loss_fp64_reference.py). Every line carries the GPU's name and power limit read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import bench  # noqa: E402
from bench_fp32_eval import gpu_info  # noqa: E402
from snag_b200 import fp32, loss as sloss  # noqa: E402
from tests import loss_fp64_reference as ref64  # noqa: E402


def step_time(layer, inputs, steps, warmup):
    streams, hidden, joint, joint_fz, wn, links, leaves = inputs

    def step():
        for t in leaves:
            t.grad = None
        loss = layer(streams, hidden, joint, joint_fz, links, wn)
        loss.backward()
        return loss

    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return round(float(np.median(ts)), 3)


def errors(emb, links):
    """(largest |nll - nll_64|, largest ||d emb - d emb_64|| / largest ||d emb_64||) of both precisions"""
    il, ir = links[:, 0].contiguous(), links[:, 1].contiguous()
    D = emb.shape[1]
    a = fp32.prep(emb, il, True, 0)[0].rows[:, :D].double()
    b = fp32.prep(emb, ir, True, 1)[0].rows[:, :D].double()
    f = ref64.icl_forward(a, b, 10.0)
    n = il.numel()
    ca = torch.full((n,), 0.5 / n, dtype=torch.float64, device=emb.device)
    nll_a, nll_b = f["nll_a"], f["nll_b"]
    out = {}
    dz = {}
    for side, (Pt, Po, Y) in (("a", (f["Pa"], f["Pb"], torch.cat([b, a], 0))), ("b", (f["Pb"], f["Pa"], torch.cat([a, b], 0)))):
        G, _, _ = ref64.icl_dlogits(Pt, Po, ca, ca, 10.0)
        dz[side] = G @ Y
        del G
    gref = torch.zeros_like(emb, dtype=torch.float64)
    gref.index_add_(0, il, ref64.normalize_bwd(emb, il, dz["a"]))
    gref.index_add_(0, ir, ref64.normalize_bwd(emb, ir, dz["b"]))
    del f, dz
    for prec in ("bf16", "fp32"):
        seen = []
        saved = sloss._IclMany

        class Spy:
            @staticmethod
            def apply(*args):
                o = saved.apply(*args)
                seen.append(o.detach())
                return o

        sloss._IclMany = Spy
        try:
            e = emb.clone().requires_grad_(True)
            sloss.icl_loss(tau=0.1, ab_weight=0.5).forward_many([e], links, precision=prec)[0].backward()
        finally:
            sloss._IclMany = saved
        nll = seen[-1][0].double()
        e_nll = float(torch.maximum((nll[0] - nll_a).abs().max(), (nll[1] - nll_b).abs().max()))
        e_grad = float((e.grad.double() - gref).norm(dim=1).max() / gref.norm(dim=1).max())
        out[prec] = {"nll_abs_err_max": e_nll, "demb_rel_err_max": e_grad}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_fp32_train_bench_n1.jsonl"))
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    lines = []
    for name in ("c1_train", "c5_train"):
        B, M, dm, _ = bench.TRAIN_WORKLOADS[name]
        streams, hidden, joint, joint_fz, wn, links, leaves = bench._train_tables(B, M, dm, dev)
        links_dev = torch.from_numpy(links).to(dev)
        inputs = (streams, hidden, joint, joint_fz, wn, links_dev, leaves)
        ms = {}
        for prec in ("bf16", "fp32"):
            layer = sloss.SnagLossLayer(tau=0.1, ab_weight=0.5, precision=prec).to(dev)
            ms[prec] = step_time(layer, inputs, args.steps, args.warmup)
            lines.append({"workload": name, "precision": prec, "B": B, "tables": f"{2 * M} x {dm} + 2 x {M * dm}",
                          "ms_per_step": ms[prec], "steps": args.steps, "warmup": args.warmup, **info})
            print(json.dumps(lines[-1]), flush=True)
        lines.append({"workload": name, "fp32_over_bf16": round(ms["fp32"] / ms["bf16"], 3), **info})
        print(json.dumps(lines[-1]), flush=True)
        links_i64 = links_dev.long()
        for tname, t in (("joint", joint), ("stream0", streams[0])):
            err = errors(t.detach().contiguous(), links_i64)
            lines.append({"workload": name, "table": tname, "D": t.shape[1], "tau": 0.1, "errors_vs_fp64": err, **info})
            print(json.dumps(lines[-1]), flush=True)
            torch.cuda.empty_cache()
        del streams, hidden, joint, joint_fz, wn, leaves, inputs
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
