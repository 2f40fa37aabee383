#!/usr/bin/env python
"""bench.py — alignment-evaluation throughput (similarity + CSLS + rank -> Hits@k / MR / MRR) on synthetic
DBP15K/FBDB15K-shaped data, the headline metric of BASELINE.json, on N GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl snag|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one full evaluation of n aligned entity pairs: gather + L2-normalise + bf16 cast of both embedding
tables, CSLS row/column neighbourhood sweeps, ground-truth scores, rank-count sweep (both directions). With N > 1
the targets are sharded over the ranks (strong scaling: the workload is fixed) and the per-row candidates /
counters are exchanged with NCCL. Rank 0 prints ONE JSON line (contract in the task statement):
  value      whole-job pairs/s, embeddings resident in HBM when the timed region starts (CUDA events, max over ranks)
  e2e        the same metric through the public API from pinned HOST buffers: H2D of the embeddings, evaluation,
             D2H of the ranks, host Hits/MR/MRR reduction — all inside the timed region
  roofline   the dominant kernel (fused tcgen05 sweep) against the measured bf16 tensor peak
  cpu_baseline  the oracle port timed on this host's cores on a bounded sample of the same workload
  parity_audit  >= 512 random sources and >= 512 random targets of the LAST timed evaluation re-scored by the oracle
             over all n partners (neighbourhood mean, ground-truth distance, rank): mismatches must be 0
  train      the metric's second half — train steps/sec of the loss-layer slice (2 + 2M icl_loss calls fwd+bwd) at
             configs[4] (B = 16 384) and at the reference's own batch (B = 3500), anchors sharded over the N ranks
  snag_step  the full SNAG training step (encoder + losses + backward) of the UNMODIFIED reference model class from
             baseline/_ref on cuda:0, stock vs with snag_b200.patch applied (rank 0)
  reference_gpu_eager  the reference's own GPU op sequence (torch-eager cuBLAS fp32 + 2n torch.sort/.item(),
             main.py:385-429; icl_loss fwd+bwd) on cuda:0 at the reference's sizes — context for a SNAG user
`--impl reference` times the CPU port alone (rank 0 only) and prints the same line with "impl": "reference".
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "align-eval entity pairs/sec (sim+CSLS+rank)"
UNIT = "pairs/s"

# name -> (n pairs, per-modality joint width D, csls k, noise sigma of the synthetic targets, description)
WORKLOADS = {
    "c4_1m": (1_000_000, 1200, 10, 6.0, "configs[3] alignment evaluation 1M x 1M entities, D=1200, CSLS k=10"),
    "c4_500k": (500_000, 1200, 10, 6.5, "configs[3] alignment evaluation 500k x 500k, D=1200, CSLS k=10"),
    "c4_200k": (200_000, 1200, 10, 7.0, "configs[3] alignment evaluation 200k x 200k, D=1200, CSLS k=10"),
    "c4_100k": (100_000, 1200, 10, 8.0, "configs[3] alignment evaluation 100k x 100k, D=1200, CSLS k=10"),
    "c1": (10_500, 1200, 10, 8.0, "configs[0] DBP15K ja_en-shaped eval, 10 500 test pairs, D=1200, CSLS k=10"),
    "c2": (10_500, 1800, 10, 8.0, "configs[1] DBP15K fr_en-shaped + surface eval, 10 500 test pairs, D=1800, CSLS k=10"),
    "c3": (10_277, 1200, 10, 8.0, "configs[2] FBDB15K-shaped eval, 10 277 test pairs, D=1200, CSLS k=10"),
}
# loss-layer slice of one training step (SURVEY 8(d)(ii)): name -> (batch B, modalities M, width per modality, description)
TRAIN_WORKLOADS = {
    "c5_train": (16384, 6, 300, "configs[4] large-batch ICL: B=16384 in-batch negatives, 6 streams x 300 (+ joint 1800), "
                                "2 + 2*6 icl_loss calls fwd+bwd per step"),
    "c2_train": (3500, 6, 300, "configs[1] DBP15K fr_en + surface: B=3500, 6 streams x 300 (+ joint 1800), 14 icl_loss calls"),
    "c1_train": (3500, 4, 300, "configs[0] DBP15K ja_en: B=3500, 4 streams x 300 (+ joint 1200), 10 icl_loss calls"),
}
TRAIN_METRIC = "train steps/sec (loss-layer slice: 2+2M icl_loss fwd+bwd)"
DEFAULT_WORKLOAD = "c4_1m"
SEED = 3408                       # the reference's scripted seed (run.sh:2)
CPU_SAMPLE_N = 8192               # bounded sample for the CPU legs: a CPU_SAMPLE_N x CPU_SAMPLE_N sub-problem (~1 s per pass on
                                  # 16 host threads: 4 passes of the cpu_baseline leg, K + W passes of the reference arm)
DUMP_ROWS = 512                   # --dump-outputs: gradient rows kept per table of a training slice (fixed, seeded choice), so
                                  # that the default line (c4_1m + c5_train + c1_train) writes about 53 MB


# ================================================================================================ helpers
def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"tensor_sustained": float(p["bf16_tflops_sustained"]), "tensor_burst": float(p["bf16_tflops"]),
                "hbm": float(p["hbm_gbs"]), "source": "MEASURED_PEAKS.json (measured)"}
    return {"tensor_sustained": 1400.0, "tensor_burst": 1590.0, "hbm": 6650.0, "source": "B200_PROFILING.md (fallback)"}


class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU while the timed region runs (NVML, 100 ms period)."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index: int):
        self.index, self.samples, self.mask, self.max_mhz = index, [], 0, None
        self.power_w, self.temp_c = [], []
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:          # NVML unavailable: report nulls rather than fail the benchmark
            self.nv = None

    def _run(self):
        while not self._stop.is_set():
            try:
                self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                self.mask |= int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.power_w.append(self.nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                self.temp_c.append(int(self.nv.nvmlDeviceGetTemperature(self.h, self.nv.NVML_TEMPERATURE_GPU)))
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self):
        s = sorted(self.samples)
        pw, tc = sorted(self.power_w), sorted(self.temp_c)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": [name for bit, name in self.REASONS.items() if self.mask & bit], "samples": len(s),
                "sm_mhz_min": (s[0] if s else None), "power_w_median": (pw[len(pw) // 2] if pw else None),
                "temp_c_max": (tc[-1] if tc else None)}


def synth_tables(n: int, d: int, sigma: float, device, chunk: int = 65536):
    """SURVEY 8(d) generator: 64 cluster centres c ~ N(0, I); x_i = N(0, I) + c_g(i); y_i = x_i + sigma N(0, I).
    Returns the joint embedding table final_emb [2n, d] fp32 (sources then targets) and the two index vectors."""
    import torch
    g = torch.Generator(device=device).manual_seed(SEED)
    centres = torch.randn((64, d), generator=g, device=device)
    emb = torch.empty((2 * n, d), dtype=torch.float32, device=device)
    for r0 in range(0, n, chunk):
        r1 = min(r0 + chunk, n)
        x = torch.randn((r1 - r0, d), generator=g, device=device)
        x += centres[torch.randint(0, 64, (r1 - r0,), generator=g, device=device)]
        emb[r0:r1] = x
        emb[n + r0:n + r1] = x + sigma * torch.randn((r1 - r0, d), generator=g, device=device)
    left = torch.arange(0, n, device=device, dtype=torch.int64)
    right = torch.arange(n, 2 * n, device=device, dtype=torch.int64)
    return emb, left, right


def dump_outputs(out_dir: str, prefix: str, arrays: dict):
    """--dump-outputs: writes every tensor of `arrays` as out_dir/<prefix>.<name>.npy, floating point as float32 and
    integers (ranks) as float64, which holds every int32 exactly."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for nm, t in arrays.items():
        t = t.detach().cpu()
        a = t.float().numpy() if t.is_floating_point() else t.to(torch.float64).numpy()
        np.save(os.path.join(out_dir, f"{prefix}.{nm}.npy"), a)


# ================================================================================================ CPU legs
def cpu_port_sample(n_s: int, d: int, k: int, sigma: float, steps: int, warmup: int):
    """Times the oracle port (oracle/snag_oracle.c, all host threads) on an n_s x n_s sub-problem of the workload."""
    import numpy as np
    from oracle import oracle
    oracle.set_threads()                 # all host cores (torchrun exports OMP_NUM_THREADS=1)
    rng = np.random.RandomState(SEED)
    centres = rng.randn(64, d).astype(np.float32)
    x = rng.randn(n_s, d).astype(np.float32) + centres[rng.randint(0, 64, n_s)]
    y = x + sigma * rng.randn(n_s, d).astype(np.float32)
    x = oracle.bf16_round(oracle.normalize_rows(x))
    y = oracle.bf16_round(oracle.normalize_rows(y))
    for _ in range(warmup):
        oracle.align_eval(x, y, True, k)
    t0 = time.perf_counter()
    for _ in range(steps):
        out = oracle.align_eval(x, y, True, k)
        oracle.metrics(out["rank_l2r"])
        oracle.metrics(out["rank_r2l"])
    dt = (time.perf_counter() - t0) / steps
    return {"value": n_s * n_s / dt, "unit": UNIT, "cores": oracle.max_threads(), "kind": "port",
            "sample": f"{n_s} x {n_s} pair sub-problem of the workload (D={d}, k={k}), {steps} timed passes, "
                      f"{dt * 1e3:.0f} ms each; oracle/snag_oracle.c with OpenMP on all host threads",
            "ms_per_step": dt * 1e3}


def reference_steps_sample(n_s: int, d: int, k: int, sigma: float):
    """The reference's literal op sequence (torch.mm, topk, per-row torch.sort + .item(), main.py:385-429) restated with
    the same torch CPU calls, timed once on a smaller sample — reported beside the port for context."""
    import numpy as np
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    rng = np.random.RandomState(SEED)
    x = torch.from_numpy(rng.randn(n_s, d).astype(np.float32))
    y = x + sigma * torch.from_numpy(rng.randn(n_s, d).astype(np.float32))
    x, y = torch.nn.functional.normalize(x), torch.nn.functional.normalize(y)
    t0 = time.perf_counter()
    x_norm = (x ** 2).sum(1).view(-1, 1)
    y_norm = (y ** 2).sum(1).view(1, -1)
    distance = torch.clamp(x_norm + y_norm - 2.0 * torch.mm(x, torch.transpose(y, 0, 1)), 0.0, np.inf)
    sim = 1 - distance
    nv1 = torch.mean(torch.topk(sim, k)[0], 1)
    nv2 = torch.mean(torch.topk(sim.t(), k)[0], 1)
    distance = 1 - ((2 * sim.t() - nv1).t() - nv2)
    mrr = 0.0
    for idx in range(n_s):
        _, indices = torch.sort(distance[idx, :], descending=False)
        rank = (indices == idx).nonzero(as_tuple=False).squeeze().item()
        mrr += 1.0 / (rank + 1)
    for idx in range(n_s):
        _, indices = torch.sort(distance[:, idx], descending=False)
        rank = (indices == idx).nonzero(as_tuple=False).squeeze().item()
        mrr += 1.0 / (rank + 1)
    dt = time.perf_counter() - t0
    return {"value": n_s * n_s / dt, "unit": UNIT, "threads": torch.get_num_threads(), "sample_n": n_s, "seconds": dt}


def run_reference(args, name, n, d, k, sigma, desc):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                      # under torchrun only rank 0 times the CPU arm; the others exit 0 without work
    n_s = min(CPU_SAMPLE_N, n)
    cb = cpu_port_sample(n_s, d, k, sigma, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32 (fp64-accumulated dots)", "data": "synthetic",
        "config": {"workload": name, "description": desc, "n_pairs": n, "width": d, "csls_k": k,
                   "sampled": f"{n_s} x {n_s} sub-problem per step"},
        "cpu_baseline": {kk: cb[kk] for kk in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ================================================================================================ GPU arm
def _bind_to_gpu_numa(index: int):
    """Pin this rank's host threads to the CPUs closest to its GPU (NVML's ideal affinity) before any pinned host buffer is
    allocated: with one rank per GPU the 8 concurrent host -> device copies of the end-to-end leg otherwise cross sockets.
    Best effort — returns the number of CPUs bound to, or None when NVML / the container does not allow it."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:                                    # noqa: BLE001
        return None


class Ctx:
    """One process per GPU: rank / device / process group of this run (torch.distributed NCCL when launched by torchrun)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus:
            if self.world == 1 and args.gpus > 1:
                raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
            raise SystemExit(f"WORLD_SIZE={self.world} does not match --gpus {args.gpus}")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.cpu_affinity = None
        self._all_cpus = os.sched_getaffinity(0)
        self.group = None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
            self.group = dist.group.WORLD
        self.peaks = load_peaks()

    def bind_host_to_gpu(self):
        """multi-rank end-to-end legs: allocate and fill the pinned host slices from the CPUs next to this rank's GPU"""
        if self.world > 1:
            self.cpu_affinity = _bind_to_gpu_numa(self.local)

    def unbind_host(self):
        if self.cpu_affinity is not None:
            os.sched_setaffinity(0, self._all_cpus)

    def barrier(self):
        import torch
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        import torch
        t = torch.tensor([x], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()


def parity_audit(X, Y, n, d, k, res, n_rows=512, n_cols=512):
    """Sampled oracle audit of one finished evaluation (rank 0, after the timed region): `n_rows` random sources against
    ALL n targets and `n_cols` random targets against ALL n sources are re-scored by oracle/snag_oracle.c (fp64
    index-order dots, the reference's fp32 chain, stable tie-break) from the very bf16 operands the GPU consumed.
    Compared bit for bit: the entity's CSLS neighbourhood mean, its ground-truth distance and its rank (the rank given
    the GPU's neighbourhood means of the other side, which the opposite sample audits)."""
    import numpy as np
    import torch
    from oracle import oracle
    oracle.set_threads()
    t0 = time.perf_counter()
    rng = np.random.RandomState(SEED + 1)
    rows = np.sort(rng.choice(n, size=min(n_rows, n), replace=False))
    cols = np.sort(rng.choice(n, size=min(n_cols, n), replace=False))
    xh = X[:n, :d].float().cpu().numpy()
    yh = Y[:n, :d].float().cpu().numpy()
    nv1, nv2 = res.nv1.cpu().numpy(), res.nv2.cpu().numpy()
    g, l2r, r2l = res.g.cpu().numpy(), res.rank_l2r.cpu().numpy(), res.rank_r2l.cpu().numpy()
    a = oracle.audit(xh[rows], yh, rows, True, k, nv2, False)
    b = oracle.audit(yh[cols], xh, cols, True, k, nv1, True)
    mism = {"nv1": int((a["nv"] != nv1[rows]).sum()), "g_rows": int((a["g"] != g[rows]).sum()),
            "rank_l2r": int((a["rank"] != l2r[rows]).sum()), "nv2": int((b["nv"] != nv2[cols]).sum()),
            "g_cols": int((b["g"] != g[cols]).sum()), "rank_r2l": int((b["rank"] != r2l[cols]).sum())}
    return {"rows": int(len(rows)), "cols": int(len(cols)), "partners_each": int(n), "mismatches": int(sum(mism.values())),
            "by_quantity": mism, "pairs_rescored": int((len(rows) + len(cols)) * n), "seconds": round(time.perf_counter() - t0, 1),
            "oracle_threads": oracle.max_threads(),
            "checked": "CSLS neighbourhood mean, ground-truth distance and rank of every sampled entity, bit-exact"}


def eval_bench(ctx, args, name):
    """The alignment-evaluation workload `name` on ctx.world GPUs -> dict of bench-line fields."""
    import torch
    import torch.distributed as dist
    from snag_b200 import evaluate, ops

    n, d, k, sigma, desc = WORKLOADS[name]
    world, rank, dev, group, peaks = ctx.world, ctx.rank, ctx.dev, ctx.group, ctx.peaks
    W, K = max(3, args.warmup), args.steps
    emb, left, right = synth_tables(n, d, sigma, dev)
    dpad = ops.round_up(d, 64)
    sweep_events = []                       # (name, start, end) per fused-sweep launch inside the timed region
    keep = {}

    def step_device():
        X, xn = ops.prep_bf16(emb, left, True)
        Y, yn = ops.prep_bf16(emb, right, True)
        keep["ops"] = (X, Y)
        return evaluate.align_ranks(X, Y, xn, yn, n, k, True, False, group)

    # ---------------------------------------------------------------- device-resident timing -> value, roofline
    res = None
    for _ in range(W):
        res = step_device()
    ctx.barrier()
    ops.SWEEP_EVENT_SINK = sweep_events
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(ctx.local) as clocks:
        ctx.barrier()
        e0.record()
        for _ in range(K):
            res = step_device()
        e1.record()
        ctx.barrier()
    ops.SWEEP_EVENT_SINK = None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, name, {"rank_l2r": res.rank_l2r, "rank_r2l": res.rank_r2l, "nv1": res.nv1,
                                               "nv2": res.nv2, "g": res.g})
    ms_per_step = ctx.max_over_ranks(e0.elapsed_time(e1) / K)
    launches_per_step = res.launches + 2
    # per-kernel durations of the fused sweeps (this rank), algorithmic flops = 2 * rows * cols * D per launch
    kern = {}
    for nm, a, b, rows, cols, _depth in sweep_events:
        kern.setdefault(nm, {"ms": [], "flops": 2.0 * rows * cols * d})["ms"].append(a.elapsed_time(b))
    kstats = {nm: {"launches": len(v["ms"]), "avg_ms": sum(v["ms"]) / len(v["ms"]),
                   "tflops": v["flops"] / (sum(v["ms"]) / len(v["ms"])) / 1e9} for nm, v in kern.items()}
    dom = max(kstats, key=lambda nm: kstats[nm]["avg_ms"] * kstats[nm]["launches"])
    # full sweeps over this rank's panel of S executed per step (from the launches themselves): 3 on the classic path,
    # 2 + 2m/n with the two-sweep CSLS path, 1 + 2m/n with the one-pass evaluation
    sweeps = sum(rows * cols for _nm, _a, _b, rows, cols, _dp in sweep_events) / K / (n * (n / world))
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(f"{dom}:{name}:{world}")
    roofline = {"bound": "tensor", "kernel": dom, "achieved": kstats[dom]["tflops"], "peak": peaks["tensor_sustained"],
                "unit": "TFLOP/s", "frac": kstats[dom]["tflops"] / peaks["tensor_sustained"], "traffic": traffic,
                "peak_source": peaks["source"] + ", bf16_tflops_sustained (kernel timed inside a long step)",
                "frac_of_burst_peak": kstats[dom]["tflops"] / peaks["tensor_burst"],
                "algorithmic_flops_per_launch": kern[dom]["flops"], "kernels": kstats,
                "sweeps_per_step": sweeps, "executed_tflops_whole_step": sweeps * 2.0 * n * n * d / world / ms_per_step / 1e9}
    out = {"ms_per_step": ms_per_step, "kernels": kstats, "roofline": roofline, "clocks": clocks.summary(),
           "launches_per_step": launches_per_step, "n": n, "d": d, "k": k, "sigma": sigma, "desc": desc, "dpad": dpad,
           "rank_sweep": res.info.get("rank_sweep", {}), "one_pass": res.info.get("one_pass"), "steps": K, "warmup": W}
    if args.profile_run:
        return out
    if world == 1 and n < evaluate.TWO_SWEEP_MIN_N:
        # reference-sized test sets: the public entry point replays the whole evaluation as ONE CUDA graph (captured on
        # the first call); time the replays — gather + normalise + cast included, as in the eager steps above
        for _ in range(3):
            evaluate.evaluate_alignment(emb, left, right, csls=True, csls_k=k)
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(K):
            o = evaluate.evaluate_alignment(emb, left, right, csls=True, csls_k=k)
        g1.record()
        torch.cuda.synchronize()
        same = bool(torch.equal(o["ranks"].rank_l2r, res.rank_l2r) and torch.equal(o["ranks"].rank_r2l, res.rank_r2l))
        out["graph_replay"] = {"ms_per_step": g0.elapsed_time(g1) / K, "cuda_graph": bool(o["ranks"].info.get("cuda_graph")),
                               "ranks_equal_eager": same,
                               "note": "evaluate_alignment(final_emb, test_left, test_right): input copy + one graph launch "
                                       "+ one 32-byte status read + host Hits/MR/MRR, per evaluation"}
    # ---------------------------------------------------------------- sampled oracle audit of the last timed evaluation
    if rank == 0 and not args.no_audit:
        X, Y = keep["ops"]
        out["parity_audit"] = parity_audit(X, Y, n, d, k, res)
    keep.clear()
    ctx.barrier()
    # ---------------------------------------------------------------- end to end from pinned host memory -> e2e
    per = (n + world - 1) // world
    c0, c1 = (0, n) if world == 1 else (rank * per, min(n, (rank + 1) * per))
    ctx.bind_host_to_gpu()
    host = torch.empty((2, max(c1 - c0, 1), d), dtype=torch.float32).pin_memory()
    host[0, :c1 - c0].copy_(emb[c0:c1])
    host[1, :c1 - c0].copy_(emb[n + c0:n + c1])
    del emb, res
    torch.cuda.empty_cache()

    def step_e2e():
        return evaluate.evaluate_alignment_host(host[0, :c1 - c0], host[1, :c1 - c0], n, c0, csls=True, csls_k=k, group=group)

    o = step_e2e()
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        o = step_e2e()
    ctx.barrier()
    dt = ctx.max_over_ranks((time.perf_counter() - t0) / K)
    out["e2e"] = {"value": n * n / dt, "unit": UNIT, "h2d_bytes_per_step": int(2 * (c1 - c0) * d * 4),
                  "d2h_bytes_per_step": int(2 * n * 4), "ms_per_step": dt * 1e3, "steps": K,
                  "streamed": bool(o.get("streamed")), "cpus_bound_to_gpu_numa": ctx.cpu_affinity,
                  "note": "per rank: H2D of its slice of both fp32 tables from pinned memory (+ NVLink all-gather of the bf16 "
                          "operands when sharded), evaluation, D2H of both rank vectors, host Hits/MR/MRR; on one GPU the "
                          "transfer is chunked and the prologue + sample pre-passes run on the chunks as they arrive"}
    ctx.unbind_host()
    m = o["l2r"]
    out["quality"] = {"hits@1_l2r": float(m.acc[0]), "hits@10_l2r": float(m.acc[1]), "mrr_l2r": m.mrr}
    del host, o
    torch.cuda.empty_cache()
    return out


def eval_line(ctx, args, name, ev):
    n, d, k = ev["n"], ev["d"], ev["k"]
    ms = ev["ms_per_step"]
    return {
        "metric": METRIC, "value": n * n / (ms * 1e-3), "unit": UNIT, "n_gpus": ctx.world, "steps": ev["steps"],
        "warmup": ev["warmup"], "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "bf16 operands, fp32 accumulate (tcgen05 kind::f16), fp32 CSLS chain, int32 ranks",
        "data": "synthetic",
        "config": {"workload": name, "description": ev["desc"], "n_pairs": n, "width": d, "padded_width": ev["dpad"],
                   "csls_k": k, "sigma": ev["sigma"], "seed": SEED, "parallelism": f"targets sharded over {ctx.world} rank(s)",
                   "l2": "inputs larger than L2 (no flush needed)" if 2 * n * ev["dpad"] * 2 > 200e6 else
                         "inputs smaller than L2; every step re-reads the fp32 table and rewrites the operands "
                         f"({2 * 2 * n * d * 4 / 1e6:.0f} MB), which exceeds and evicts L2"},
        "clocks": ev["clocks"], "e2e": ev.get("e2e"), "gpu_launches": ev["launches_per_step"] * ev["steps"],
        "roofline": ev["roofline"], "quality": ev.get("quality"),
        "algorithmic_tflops": 2.0 * n * n * d / (ms * 1e-3) / 1e12, "rank_sweep": ev["rank_sweep"], "one_pass": ev.get("one_pass"),
        "parity_audit": ev.get("parity_audit"), "graph_replay": ev.get("graph_replay"),
    }


# ================================================================================================ training slice
def _train_tables(B, M, dm, device, seed=SEED):
    """Stand-ins for the encoder outputs of one step (model/SNAG.py:101-102): M modality embeddings and M hidden-state
    embeddings [N, dm], two joint embeddings [N, M*dm], modality weights [N, M]; N = 2B + 1000 entities, B random links."""
    import numpy as np
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    n_ent = 2 * B + 1000
    mk = lambda w: torch.randn((n_ent, w), generator=g, device=device).requires_grad_(True)
    present = [True] * M + [False] * (6 - M)              # (gph, rel, att, img, name, char): surface streams last
    streams = [mk(dm) if p else None for p in present]
    hidden = [mk(dm) if p else None for p in present]
    joint, joint_fz = mk(M * dm), mk(M * dm)
    wn = torch.softmax(torch.randn((n_ent, 6), generator=g, device=device), 1).requires_grad_(True)
    rng = np.random.RandomState(seed)
    links = np.stack([rng.permutation(n_ent // 2)[:B], n_ent // 2 + rng.permutation(n_ent // 2)[:B]], 1).astype(np.int32)
    leaves = [t for t in streams + hidden + [joint, joint_fz, wn] if t is not None]
    return streams, hidden, joint, joint_fz, wn, links, leaves


def cpu_icl_sample(B_s, M, dm, steps, B_full=None):
    """The reference's icl_loss op sequence (model/SNAG_loss.py:58-128: normalise, 4 matmuls, -1e9 self mask, concat,
    log_softmax against one-hot labels, weighted mean) restated with the same torch CPU calls, forward + backward, for
    the 2 + 2M calls of one step at batch B_s, all host threads."""
    import torch
    import torch.nn.functional as F
    torch.set_num_threads(os.cpu_count() or 1)
    g = torch.Generator().manual_seed(SEED)
    n_ent = 2 * B_s + 100
    links = torch.stack([torch.randperm(n_ent // 2, generator=g)[:B_s], n_ent // 2 + torch.randperm(n_ent // 2, generator=g)[:B_s]], 1)

    def icl(emb, w):
        z = F.normalize(emb, dim=1)
        a, b = z[links[:, 0]], z[links[:, 1]]
        eye = torch.eye(B_s) * 1e9
        lab = F.one_hot(torch.arange(B_s), 2 * B_s).float()
        la = torch.cat([a @ b.t(), a @ a.t() - eye], 1) / 0.1
        lb = torch.cat([b @ a.t(), b @ b.t() - eye], 1) / 0.1
        wt = torch.ones(B_s) if w is None else torch.min(w[links[:, 0]], w[links[:, 1]])
        xa = -(wt * (lab * F.log_softmax(la, 1)).sum(1)).sum() / B_s
        xb = -(wt * (lab * F.log_softmax(lb, 1)).sum(1)).sum() / B_s
        return 0.5 * xa + 0.5 * xb

    embs = [torch.randn((n_ent, dm), generator=g).requires_grad_(True) for _ in range(2 * M)]
    joints = [torch.randn((n_ent, M * dm), generator=g).requires_grad_(True) for _ in range(2)]
    w = torch.rand((n_ent,), generator=g)
    t0 = time.perf_counter()
    for _ in range(steps):
        tot = sum(icl(e, w if i < M else None) for i, e in enumerate(embs)) + sum(icl(j, None) for j in joints)
        tot.backward()
    dt = (time.perf_counter() - t0) / steps
    scale = 1.0 if not B_full else (B_s / float(B_full)) ** 2          # every term of the step is O(B^2 D)
    return {"value": scale / dt, "unit": "steps/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"one step at batch {B_s} ({2 + 2 * M} icl_loss calls fwd+bwd, the reference's torch op sequence on CPU "
                      f"tensors), {steps} timed step(s), {dt * 1e3:.0f} ms each, scaled by (B_s/B)^2 = {scale:.4g} to the "
                      f"workload's batch (the step is O(B^2 D))"}


def train_bench(ctx, args, name, cpu_leg=True):
    """The loss-layer slice `name` (2 + 2M icl_loss calls, forward + backward) on ctx.world GPUs -> bench-line fields."""
    import numpy as np
    import torch
    from snag_b200 import loss as sloss, ops

    B, M, dm, desc = TRAIN_WORKLOADS[name]
    world, rank, dev, group, peaks = ctx.world, ctx.rank, ctx.dev, ctx.group, ctx.peaks
    W, K = max(3, args.warmup), args.steps
    streams, hidden, joint, joint_fz, wn, links, leaves = _train_tables(B, M, dm, dev)
    layer = sloss.SnagLossLayer(tau=0.1, ab_weight=0.5).to(dev)       # --awloss 0 (config.py:114): the reference's default
    links_pinned = torch.from_numpy(links).pin_memory()
    links_dev = links_pinned.to(dev)

    def eager_step():
        for t in leaves:
            t.grad = None
        loss = layer(streams, hidden, joint, joint_fz, links_dev, wn)
        loss.backward()
        return loss

    def measure(grads_mode):
        """Timed region of the slice with the gradient exchange `grads_mode` ("local": every rank returns the rows of
        dL/d emb of the anchors it owns, zeros elsewhere — the sum over ranks is the gradient, which the data-parallel
        gradient all-reduce of a replicated encoder completes anyway; "gather": the owned rows are all-gathered so that
        every rank returns the full gradient, as an unsharded call would)."""
        if group is not None:
            layer.distribute(group, grads=grads_mode)
        graph_note = None
        for _ in range(3):
            eager_step()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.barrier()
        a.record()
        for _ in range(K):
            eager_step()
        b.record()
        ctx.barrier()
        eager_ms = ctx.max_over_ranks(a.elapsed_time(b) / K)
        # Whole-step CUDA graph: every entry point of libsnag_b200.so only enqueues on the stream it is given, and NCCL's
        # all-gathers are capturable, so the sharded step replays as one graph launch as well (at the reference's batch
        # sizes the eager step is launch bound). Every rank must take the same path: agree on the outcome of the capture.
        use_graph = not args.no_graph
        graphed = None
        if use_graph:
            ok = 1.0
            try:
                from snag_b200.graphs import GraphedStep
                graphed = GraphedStep(lambda: layer(streams, hidden, joint, joint_fz, links_dev, wn), leaves)
            except Exception as exc:                          # noqa: BLE001 — reported on the bench line, eager numbers stand
                ok, graph_note = 0.0, f"graph capture failed on rank {rank}: {type(exc).__name__}: {exc}"[:300]
            if -ctx.max_over_ranks(-ok) < 1.0:
                use_graph, graphed = False, None
                graph_note = graph_note or "graph capture failed on another rank"

        def step(from_host):
            if from_host:                                       # this step's batch arrives from pinned host memory
                links_dev.copy_(links_pinned, non_blocking=True)
            loss = graphed() if use_graph else eager_step()
            return loss.item() if from_host else loss

        for _ in range(W):
            step(False)
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(ctx.local) as clocks:
            ctx.barrier()
            e0.record()
            for _ in range(K):
                loss = step(False)
            e1.record()
            ctx.barrier()
        if args.dump_outputs and grads_mode == "local" and rank == 0:
            rows = torch.from_numpy(np.sort(np.random.RandomState(SEED + 2).choice(wn.shape[0], DUMP_ROWS, replace=False)))
            named = [(f"stream{m}", t) for m, t in enumerate(streams)] + [(f"hidden{m}", t) for m, t in enumerate(hidden)]
            named += [("joint", joint), ("joint_fz", joint_fz), ("weight_norm", wn)]
            dump_outputs(args.dump_outputs, name, {"loss": loss.reshape(1), **{f"grad_{nm}": t.grad[rows.to(dev)]
                                                                                for nm, t in named if t is not None}})
        ms = ctx.max_over_ranks(e0.elapsed_time(e1) / K)
        # end to end: the step's input (the batch of links) comes from pinned host memory, the loss goes back to the host
        step(True)
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            lv = step(True)
        ctx.barrier()
        dt = ctx.max_over_ranks((time.perf_counter() - t0) / K)
        del graphed
        return {"ms": ms, "eager_ms": eager_ms, "use_graph": use_graph, "graph_note": graph_note, "clocks": clocks.summary(),
                "e2e_s": dt, "loss": lv}

    gather = measure("gather") if group is not None else None
    head = measure("local")
    ms_per_step, eager_ms, use_graph, graph_note = head["ms"], head["eager_ms"], head["use_graph"], head["graph_note"]
    # per-kernel CUDA events cannot be recorded into a replayed graph: time the sweeps of K eager steps of the same work
    events = []
    ops.SWEEP_EVENT_SINK = events
    for _ in range(K):
        eager_step()
    torch.cuda.synchronize()
    ops.SWEEP_EVENT_SINK = None
    kern = {}
    for nm, ea, eb, rows, cols, depth in events:
        e = kern.setdefault(nm, {"ms": 0.0, "flops": 0.0, "launches": 0})
        e["ms"] += ea.elapsed_time(eb)
        e["flops"] += 2.0 * rows * cols * depth
        e["launches"] += 1
    kstats = {nm: {"launches_per_step": v["launches"] // K, "ms_per_step": v["ms"] / K, "tflops": v["flops"] / v["ms"] / 1e9}
              for nm, v in kern.items()}
    dom = max(kstats, key=lambda nm: kstats[nm]["ms_per_step"])
    n_calls = 2 + 2 * M
    d_sum = 2 * M * dm + 2 * M * dm                        # sum of the contraction widths over the calls
    alg_fwd = 6.0 * B * B * d_sum                          # SURVEY 8(d): 3 distinct B x B x D contractions per call
    alg_bwd = 14.0 * B * B * d_sum
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(f"{dom}:{name}:{world}")
    roofline = {"bound": "tensor", "kernel": dom, "achieved": kstats[dom]["tflops"], "peak": peaks["tensor_burst"],
                "unit": "TFLOP/s", "frac": kstats[dom]["tflops"] / peaks["tensor_burst"], "traffic": traffic,
                "peak_source": peaks["source"] + ", bf16_tflops (burst: launches of a few ms, timed alone with CUDA events)",
                "kernels": kstats, "note": "flops counted on the padded contraction width the kernel executes",
                "algorithmic_flops_per_step": alg_fwd + alg_bwd,
                "algorithmic_tflops_whole_step": (alg_fwd + alg_bwd) / world / ms_per_step / 1e9}
    dt, lv = head["e2e_s"], head["loss"]
    out = {"metric": TRAIN_METRIC, "value": 1e3 / ms_per_step, "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": W,
           "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "bf16 operands, fp32 accumulate (tcgen05 kind::f16), fp32 softmax statistics",
           "data": "synthetic",
           "config": {"workload": name, "description": desc, "batch": B, "modalities": M, "width": dm, "tau": 0.1,
                      "icl_calls_per_step": n_calls, "parallelism": f"anchors sharded over {world} rank(s)", "awloss": 0,
                      "grads": "n/a (one rank)" if group is None else
                               "local: each rank returns the rows of dL/d emb of its own anchors; their sum over the ranks is the "
                               "gradient (what a data-parallel trainer's gradient all-reduce forms) — the all-gathered form is "
                               "timed beside it as grads_gather",
                      "cuda_graph": use_graph, "graph_note": graph_note, "eager_ms_per_step": eager_ms,
                      "l2": "every step rewrites the bf16 operands and gradients (> L2) between launches"},
           "clocks": head["clocks"],
           "e2e": {"value": 1.0 / dt, "unit": "steps/s", "h2d_bytes_per_step": int(links_pinned.numel() * 4),
                   "d2h_bytes_per_step": 4, "ms_per_step": dt * 1e3, "loss": lv},
           "gpu_launches": (sum(v["launches"] for v in kern.values()) // K + 4 * n_calls) * K,
           "roofline": roofline}
    if gather is not None:
        out["grads_gather"] = {"ms_per_step": gather["ms"], "value": 1e3 / gather["ms"], "unit": "steps/s",
                               "eager_ms_per_step": gather["eager_ms"], "cuda_graph": gather["use_graph"],
                               "e2e_ms_per_step": gather["e2e_s"] * 1e3,
                               "what": "the same step with the owned gradient rows all-gathered: every rank returns the full "
                                       "dL/d emb of all 2 + 2M tables"}
    if cpu_leg and rank == 0:
        out["cpu_baseline"] = cpu_icl_sample(min(B, 1024), M, dm, 1, B)
    del layer, streams, hidden, joint, joint_fz, wn, leaves
    torch.cuda.empty_cache()
    return out


# ================================================================================================ context legs (rank 0)
def reference_gpu_eager(dev, n=10500, d=1200, k=10, sigma=8.0, B=3500, M=4, dm=300):
    """What a SNAG user runs today on the same GPU (main.py:517-519 puts the model on one GPU): the reference's literal
    evaluation sequence — pairwise_distances (src/utils.py:202-218), csls_sim (:417-435), then 2n x (torch.sort of a
    row / column + .item()), main.py:385-429 — and its icl_loss forward + backward (model/SNAG_loss.py:58-128) for the
    2 + 2M calls of one step, all in torch-eager fp32 on CUDA (cuBLAS SGEMM, TF32 off as in the reference). Imported
    from the unmodified reference when baseline/_ref travels with the repo, restated with the same torch calls
    otherwise. Context only: it is a GPU number of the reference, not the CPU baseline the contract asks for."""
    import numpy as np
    import torch
    import torch.nn.functional as F
    out = {}
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        from baseline import harness
        harness.load_reference()
        import model.SNAG_loss as ref_loss
        import src.utils as ref_utils
        pd, cs, icl_cls, src = ref_utils.pairwise_distances, ref_utils.csls_sim, ref_loss.icl_loss, "baseline/_ref (unmodified reference functions)"
    except Exception:                      # noqa: BLE001 — no reference checkout on this machine: same torch calls, restated
        def pd(x, y):
            xn, yn = (x ** 2).sum(1).view(-1, 1), (y ** 2).sum(1).view(1, -1)
            return torch.clamp(xn + yn - 2.0 * torch.mm(x, y.t()), 0.0, np.inf)

        def cs(sim, kk):
            nv1, nv2 = torch.mean(torch.topk(sim, kk)[0], 1), torch.mean(torch.topk(sim.t(), kk)[0], 1)
            return (2 * sim.t() - nv1).t() - nv2
        icl_cls, src = None, "restated torch calls (no reference checkout here)"
    emb, left, right = synth_tables(n, d, sigma, dev)
    torch.cuda.synchronize()

    def eval_once():
        fe = F.normalize(emb)
        distance = pd(fe[left], fe[right])
        distance = 1 - cs(1 - distance, k)
        mrr = 0.0
        for idx in range(n):
            _, indices = torch.sort(distance[idx, :], descending=False)
            rank_ = (indices == idx).nonzero(as_tuple=False).squeeze().item()
            mrr += 1.0 / (rank_ + 1)
        for idx in range(n):
            _, indices = torch.sort(distance[:, idx], descending=False)
            rank_ = (indices == idx).nonzero(as_tuple=False).squeeze().item()
            mrr += 1.0 / (rank_ + 1)
        return mrr

    eval_once() if n <= 4096 else None
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eval_once()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    out["eval"] = {"value": n * n / dt, "unit": UNIT, "seconds": dt, "n_pairs": n, "width": d, "csls_k": k,
                   "what": "F.normalize + pairwise_distances + csls_sim + 2n x (torch.sort + .item()), fp32, cuda:0"}
    del emb
    torch.cuda.empty_cache()
    if icl_cls is not None:
        streams, hidden, joint, joint_fz, wn, links, leaves = _train_tables(B, M, dm, dev)
        crit = icl_cls(tau=0.1, ab_weight=0.5, n_view=2)
        cols = (3, 2, 1, 0, 4, 5)

        def step():
            for t in leaves:
                t.grad = None
            w = wn * wn.shape[1]
            tot = crit(joint, links) + crit(joint_fz, links)
            tot = tot + sum(crit(e, links, weight_norm=w[:, c]) for e, c in zip(streams, cols) if e is not None)
            tot = tot + sum(crit(h, links) for h in hidden if h is not None)
            tot.backward()
            return tot
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps = 5
        for _ in range(reps):
            step().item()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / reps
        out["train_slice"] = {"value": 1.0 / dt, "unit": "steps/s", "ms_per_step": dt * 1e3, "batch": B, "modalities": M,
                              "what": f"{2 + 2 * M} reference icl_loss calls fwd+bwd (unmodified class), fp32, cuda:0"}
    out["source"] = src
    return out


def snag_full_step(dev, n_side=19797, n_links=15000, batch=3500, steps=5):
    """SURVEY 8(d)(ii): the full training step of the UNMODIFIED reference SNAG model (GAT encoder, modality
    projections, fusion transformer, 2 + 2M icl_loss calls, backward, AdamW) at the C1 shape — N = 39 594 entities,
    4 500 seed links, B = 3500, per-modality width 300 — on cuda:0, first stock, then with snag_b200.patch applied
    (new model instance, same state dict). Data: baseline/harness.py's synthetic graph pair in the reference's own
    file format. Returns None when the reference does not travel with the repo (baseline/_ref)."""
    import logging
    import shutil
    import tempfile
    import numpy as np
    import torch
    from baseline import harness
    if harness.ref_root() is None:
        return None
    from snag_b200 import patch as spatch
    root = harness.load_reference()
    tmp = tempfile.mkdtemp(prefix="snag_bench_")
    cwd = os.getcwd()
    out = {}
    try:
        harness.write_dataset(tmp, n_side=n_side, n_links=n_links, img_dim=2048)
        argv = harness.main_argv(tmp, epochs=1, batch_size=batch)
        for key, val in (("--hidden_units", "300,300,300"), ("--attr_dim", "300"), ("--img_dim", "300"), ("--name_dim", "300"),
                         ("--char_dim", "300"), ("--hidden_size", "300"), ("--intermediate_size", "400")):
            argv[argv.index(key) + 1] = val
        cfgs = harness.parse_args(argv)
        cfgs.device = dev
        os.chdir(root)
        import importlib
        import main as ref_main
        ref_snag = importlib.import_module("model.SNAG")             # the module (model/__init__ re-exports the class under the same name)
        logger = logging.getLogger("snag_bench_ref")
        logger.setLevel(logging.WARNING)
        runner = ref_main.Runner(cfgs, None, logger)
        train_ill = np.asarray(runner.train_ill, dtype=np.int32)
        batch_links = train_ill[:batch]

        def time_steps(model, optim):
            model.train()
            model.update_noise()

            def one():
                loss, _ = model(batch_links)
                loss.backward()
                torch.nn.utils.clip_grad_norm_(model.parameters(), cfgs.clip)
                optim.step()
                model.zero_grad(set_to_none=True)
                return loss
            for _ in range(2):
                one()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                lv = one().item()
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / steps, lv

        state = {k_: v.clone() for k_, v in runner.model.state_dict().items()}
        dt_ref, loss_ref = time_steps(runner.model, runner.optimizer)
        spatch.patch(ref_main)
        model_p = ref_snag.SNAG(runner.KGs, cfgs).cuda()
        model_p.load_state_dict(state)
        from src.utils import set_optim
        optim_p, _ = set_optim(cfgs, [model_p], [], [])              # the reference's parameter groups (src/utils.py:24-81)
        dt_p, loss_p = time_steps(model_p, optim_p)
        out = {"entities": 2 * n_side, "batch": int(batch_links.shape[0]), "modalities": 4, "width": 300,
               "stock_ms_per_step": dt_ref * 1e3, "patched_ms_per_step": dt_p * 1e3, "stock_steps_per_s": 1.0 / dt_ref,
               "patched_steps_per_s": 1.0 / dt_p, "speedup": dt_ref / dt_p, "stock_loss": loss_ref, "patched_loss": loss_p,
               "what": "update_noise once, then model(batch) + backward + clip + AdamW per step, wall clock with the loss "
                       "read back every step; stock = unmodified reference on cuda:0 (fp32 torch eager)"}
    finally:
        try:
            spatch.unpatch()
        finally:
            os.chdir(cwd)
            shutil.rmtree(tmp, ignore_errors=True)
    return out


def run_snag(args, name):
    ctx = Ctx(args)
    ev = eval_bench(ctx, args, name)
    if args.profile_run:
        if ctx.rank == 0:
            print(json.dumps({"profile_run": True, "workload": name, "ms_per_step": ev["ms_per_step"], "kernels": ev["kernels"]}), flush=True)
        ctx.close()
        return
    line = eval_line(ctx, args, name, ev) if ctx.rank == 0 else None
    n, d, k, sigma = ev["n"], ev["d"], ev["k"], ev["sigma"]
    # the metric's second half: train steps/sec of the loss-layer slice at every N (anchors sharded over the ranks)
    train = {}
    if not args.no_train:
        for tname in ("c5_train", "c1_train"):
            train[tname] = train_bench(ctx, args, tname, cpu_leg=(ctx.world == 1))
    if ctx.rank == 0:
        line["train"] = {t: {kk: v[kk] for kk in ("metric", "value", "unit", "ms_per_step", "scaling", "config", "e2e", "roofline",
                                                    "gpu_launches", "clocks") + (("cpu_baseline",) if "cpu_baseline" in v else ()) +
                             (("grads_gather",) if "grads_gather" in v else ())}
                         for t, v in train.items()}
        n_s = min(CPU_SAMPLE_N, n)
        cb = cpu_port_sample(n_s, d, k, sigma, 3, 1)
        line["cpu_baseline"] = {kk: cb[kk] for kk in ("value", "unit", "cores", "kind", "sample")}
        line["reference_literal_steps"] = reference_steps_sample(min(2048, n), d, k, sigma)
        if not args.no_context:
            import contextlib
            # the reference print()s its progress ("loading raw data...") — keep stdout to the ONE JSON line
            with contextlib.redirect_stdout(sys.stderr):
                try:
                    line["snag_step"] = snag_full_step(ctx.dev)
                except Exception as exc:                  # noqa: BLE001 — a context leg must not take the headline down
                    line["snag_step"] = {"error": f"{type(exc).__name__}: {exc}"[:400]}
                try:
                    line["reference_gpu_eager"] = reference_gpu_eager(ctx.dev)
                except Exception as exc:                  # noqa: BLE001
                    line["reference_gpu_eager"] = {"error": f"{type(exc).__name__}: {exc}"[:400]}
        print(json.dumps(line), flush=True)
    ctx.close()


def run_train(args, name):
    B, M, dm, desc = TRAIN_WORKLOADS[name]
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            cb = cpu_icl_sample(min(B, 2048), M, dm, max(1, args.steps), B)
            print(json.dumps({"impl": "reference", "metric": TRAIN_METRIC, "value": cb["value"], "unit": "steps/s",
                              "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / cb["value"],
                              "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                              "config": {"workload": name, "description": desc, "sampled": cb["sample"]}, "cpu_baseline": cb,
                              "e2e": {"value": cb["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                              "gpu_launches": 0}), flush=True)
        return
    ctx = Ctx(args)
    out = train_bench(ctx, args, name)
    if ctx.rank == 0:
        print(json.dumps(out), flush=True)
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3,
                    help="steps of every GPU timed loop: the device-resident steps, the end-to-end steps and the CUDA-graph "
                         "replays of the small evaluations (a short window makes the last two noisier)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=os.environ.get("SNAG_BENCH_WORKLOAD", DEFAULT_WORKLOAD), choices=sorted(WORKLOADS) + sorted(TRAIN_WORKLOADS))
    ap.add_argument("--impl", default="snag", choices=["snag", "reference"])
    ap.add_argument("--no-graph", action="store_true", help="training slice: run the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-train", action="store_true", help="evaluation workloads: skip the train blocks of the line")
    ap.add_argument("--no-audit", action="store_true", help="evaluation workloads: skip the sampled oracle audit")
    ap.add_argument("--no-context", action="store_true", help="skip the snag_step / reference_gpu_eager context legs")
    ap.add_argument("--profile-run", action="store_true",
                    help="only the device-resident timed region (for runs under ncu); e2e and CPU legs are skipped")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of each GPU workload computed as DIR/<workload>.<name>.npy: the rank "
                         "vectors, CSLS neighbourhood means and ground-truth distances of an evaluation; the loss and a "
                         f"fixed sample of {DUMP_ROWS} rows of every input gradient of a training slice. Rank 0 writes what it "
                         "received: with --gpus N > 1 a training gradient holds only the rows of rank 0's own anchors "
                         "(zeros elsewhere), not the full gradient")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "snag":
        ap.error("--dump-outputs writes the outputs of --impl snag")
    if args.workload in TRAIN_WORKLOADS:
        run_train(args, args.workload)
        return
    n, d, k, sigma, desc = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, args.workload, n, d, k, sigma, desc)
    else:
        run_snag(args, args.workload)


if __name__ == "__main__":
    main()
