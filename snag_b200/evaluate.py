"""Alignment evaluation: source x target similarity, CSLS correction, ranking into Hits@k / MR / MRR.

Host-side mirror of the reference's evaluation interface
  - pairwise_distances(x, y=None)          SNAG_MMEA/src/utils.py:202-218
  - csls_sim(sim_mat, k)                   SNAG_MMEA/src/utils.py:417-435
  - the ranking body of Runner._test       SNAG_MMEA/main.py:379-436
on top of the fused tcgen05 sweeps of libsnag_b200.so. The n x n matrix is never materialised on the
fused path (`align_ranks`); the two drop-ins that must return a matrix do materialise it.

Sharded evaluation: targets are split into contiguous shards, one per rank (one process per GPU); every
rank holds both embedding tables and sweeps all sources against its own targets. Per sweep there is one
exchange step (NCCL all-gather of per-row CSLS candidates / neighbourhood means / column counters, all-reduce
of the integer row counters). Integer counters make the result identical for any number of ranks.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
import torch

from . import ops as _cuda_ops
from ._lib import KT, SnagError
from .ops import round_up

TOP_K = (1, 10, 50)   # main.py:380


# =================================================================================================
# fused path
# =================================================================================================
@dataclass
class AlignRanks:
    rank_l2r: torch.Tensor            # int32 [n]  0-based position of target i in the sorted row i
    rank_r2l: torch.Tensor            # int32 [n]  0-based position of source j in the sorted column j
    nv1: torch.Tensor | None          # fp32 [n]   CSLS row neighbourhood means
    nv2: torch.Tensor | None          # fp32 [n]   CSLS column neighbourhood means
    g: torch.Tensor                   # fp32 [n]   distance of the ground-truth pair
    top3_idx: torch.Tensor | None = None   # int32 [n,3] pair ids of the 3 nearest targets per source
    top3_val: torch.Tensor | None = None
    launches: int = 0                 # kernels of libsnag_b200.so launched by this rank
    info: dict = field(default_factory=dict)


def shard_bounds(n: int, world: int, rank: int, align: int = 256) -> tuple[int, int]:
    """Contiguous target shard [c0, c1) of `rank`; every shard but the last has `per` = ceil(n/world) rounded
    up to `align` targets (column tiles are 256 wide), trailing ranks may own nothing."""
    per = round_up((n + world - 1) // world, align)
    c0 = min(rank * per, n)
    c1 = min(c0 + per, n)
    return c0, c1


TWO_SWEEP_MIN_N = 65536     # below this the sample pre-pass costs more than the sweep it saves
SAMPLE_MAX = 32768          # largest pre-pass sample (sources and targets each)


def two_sweep_plan(n: int, k: int, n_targets: int | None = None, n_ctas: int = 148) -> tuple[int, int] | None:
    """(sample size m, candidate-stream capacity per CTA) of the two-sweep CSLS path, or None when n is too small.
    A random sample of m sources leaves on average k*n/m candidates per target (for any data distribution: the
    rows are exchangeable), i.e. k*n*n_targets/m in total for the n_targets this rank owns (default: all n), spread
    over its n_ctas persistent CTAs in proportion to the tiles they process; each CTA's stream holds twice its even
    share. m depends on n alone, so every rank of a sharded evaluation draws the same sample."""
    if n < TWO_SWEEP_MIN_N:
        return None
    m = min(max(round_up(n // 16, 256), 8192), SAMPLE_MAX)
    nt = n if n_targets is None else max(1, int(n_targets))
    cap = round_up(int(2.0 * k * n / m * nt / max(1, n_ctas)) + 4096, 1024)
    return m, cap


# One-pass evaluation (n >= TWO_SWEEP_MIN_N, CSLS, no prediction file): the main sweep also streams out every element that
# may count towards a rank, judged after the neighbourhood means are final — the second sweep over S is not needed.
ONE_PASS = True
ONE_PASS_GAMMA = 1.5                 # safety factor on the sample -> population extrapolation of the guessed upper bounds
ONE_PASS_STREAM_PER_TARGET = 1024    # rank-stream entries provided per owned target (both directions together)
ONE_PASS_EXHAUSTIVE_MAX = 32         # up to this many entities whose guess failed are recounted with fp64 dots ...
ONE_PASS_RECOUNT_MAX_FRAC = 0.8      # ... more by tensor-core sweeps over the gathered sub-panels (a fraction failed_rows / n +
                                     # failed_cols / n_targets of a sweep), unless that exceeds this much of sweep 2
_ONE_PASS_CAP: dict = {}             # (n, ns, k, dpad) -> per-CTA stream capacity that was enough last time

_SAMPLES: dict = {}


def _sample_rows(n: int, m: int, dev):
    """The two fixed random samples (of sources, of targets) the pre-passes use: m sorted row ids each, drawn once per
    (n, m, device) from a seeded CPU generator — the same on every rank, and not re-drawn on every evaluation (a
    torch.randperm of 10^6 on the host costs ~15 ms, during which the GPU would sit idle)."""
    key = (n, m, str(dev))
    if key not in _SAMPLES:
        gsel = torch.Generator(device="cpu").manual_seed(3408)
        sel_h = torch.randperm(n, generator=gsel)[:m].sort()[0]
        selc_h = torch.randperm(n, generator=gsel)[:m].sort()[0]
        if len(_SAMPLES) > 16:
            _SAMPLES.clear()
        _SAMPLES[key] = (sel_h.to(dev), selc_h.to(dev), sel_h, selc_h)
    return _SAMPLES[key][:2]


def _sample_rows_host(n: int, m: int, dev):
    """The same two samples as host tensors (for gathering sampled rows out of host memory)."""
    _sample_rows(n, m, dev)
    return _SAMPLES[(n, m, str(dev))][2:]


LAZY_NORM2_BOUND = 1.02     # squared row norm the sync-free path assumes (F.normalize'd rows rounded to bf16: 1 +- 4e-3)


def _align_ranks_steps(be, X, Y, xn, yn, n: int, csls_k: int, use_csls: bool, want_top3: bool, world: int, rank: int,
                       two_sweep: bool = True, lazy: bool = False, one_pass: bool | None = None, pre: dict | None = None):
    """Generator form of the sharded evaluation. Yields ("all_gather", t) / ("all_reduce", t) whenever the ranks
    must exchange data and receives the collective's result (all_gather: tensor with a new leading dim of size
    world; all_reduce: the elementwise sum). Returning through StopIteration.value keeps the data path identical
    for torch.distributed (NCCL / gloo) and for the in-process lockstep simulator used by the tests.
    `be` is the kernel backend (snag_b200.ops).
    lazy (single rank, three-sweep path only): nothing in here synchronises with the host — the tolerances assume
    nearly-unit rows (LAZY_NORM2_BOUND) and the device-side counters that normally steer retries are returned in
    info["pending"] for align_ranks to check once, after everything has been enqueued.
    pre (single rank, two-sweep sizes): {"cand_r": [n, KT], "cand_s": [n, KT]} — the merged candidate lists of the two
    sample pre-passes when the caller already ran them (evaluate_alignment_host does, chunk by chunk, while the tables
    are still arriving from the host); they must come from the samples _sample_rows(n, m, device) names."""
    dev = X.device
    launches = 0
    kw = dict(norm_bound=LAZY_NORM2_BOUND ** 0.5, lazy=True) if lazy else {}
    if lazy:
        be.LAST_TOPK_INFO.clear()                  # the info entries below must be this evaluation's device counters
    c0, c1 = shard_bounds(n, world, rank)
    ns = c1 - c0                                   # targets owned by this rank
    per = shard_bounds(n, world, 0)[1]             # padded shard size used for the gathers
    Ys = Y[c0:c1] if ns > 0 else None
    yns = yn[c0:c1] if ns > 0 else None

    nv1 = nv2 = None
    if use_csls:
        # Sweep 1 selects, per source and per target, the KT partners with the largest tensor-core score and remembers
        # WHO they are; the neighbourhood means are then computed from those candidates with the canonical arithmetic
        # (ops.topk_rescore), so nv1 / nv2 equal the oracle's bit for bit whatever the accumulation order of the MMAs.
        col_val = col_idx = col_bound = None
        plan2 = two_sweep_plan(n, csls_k, ns, be.num_sms()) if (two_sweep and hasattr(be, "eval_rowcoltopk")) else None
        part = pidx = None
        one = None          # state of the one-pass evaluation (relaxed constants, rank streams) or None
        if plan2 is not None:
            # two-sweep path: sample pre-passes bound every target's k-th best and every source's KT-th best from
            # below; the main sweep then builds the row lists from those bounds and collects, per target, every source
            # at or above its bound, so the swapped sweep is not needed.
            m, cap = plan2
            if one_pass is None:
                one_pass = ONE_PASS
            # largest squared row norm: the fused sweep's fp16x2 pre-filter (and with it the one-pass evaluation) is for
            # L2-normalised rows; anything else takes the fp32 form of the two-sweep path
            nrm2 = float(torch.maximum(xn[:n].max(), yn[:n].max()).item())
            if one_pass and not want_top3 and hasattr(be, "eval_onepass") and nrm2 <= be.HALF_PREFILTER_NORM2_MAX:
                import math
                eps = be.rank_band_eps(xn, yn, X.shape[1])
                one = {"eps": eps, "delta": 2.0 * eps + 2e-6,
                       "shift": ONE_PASS_GAMMA * math.log(max(n / m, 1.0))}
                # canonical c of every ground-truth pair: the one neighbour of an entity known before the sweep
                one["c_diag"] = 1.0 - be.pair_score(X, Y, n, xn, yn, None, None, False)
                launches += 1
            sel, selc = _sample_rows(n, m, dev)
            # Row bounds: the KT-th best of a source over a random sample of ALL targets can only be lower than its
            # KT-th best overall, so lists seeded with it lose nothing and skip their warm-up. (A sample of 8192 instead
            # of 32768 targets was measured at 4 ranks: pre-pass 21 ms cheaper, sweep 88 ms slower.) The sample is
            # global and identical on every rank; each rank computes the bounds of its slice of the sources and the
            # slices are all-gathered, so this pre-pass shrinks with the number of ranks like the sweeps do.
            Yc, ync = (Y.index_select(0, selc), yn.index_select(0, selc)) if pre is None else (None, None)
            per_r = (n + world - 1) // world
            a0, a1 = min(rank * per_r, n), min((rank + 1) * per_r, n)
            nrow = 3 if one is not None else 1          # rows of the exchanged block: rowthr (, lo1, hi1)
            thr_loc = torch.full((nrow, per_r), float("-inf"), dtype=torch.float32, device=dev)
            if a1 > a0:
                if pre is not None:
                    part_r, cand_r = None, pre["cand_r"]
                else:
                    part_r = be.eval_rowtopk(X[a0:a1], Yc, xn[a0:a1], ync, a1 - a0, m)
                    _, cand_r = be.topk_merge_mean(part_r, csls_k, want_nv=False, want_cand=True)
                    launches += 2
                thr_loc[0, :a1 - a0] = cand_r[:, 0] - 2e-6             # lists are ascending: [0] is the KT-th largest
                if one is not None:
                    lo1, hi1 = be.spec_bounds(cand_r, one["c_diag"][a0:a1].contiguous(), csls_k, one["shift"], one["delta"])
                    thr_loc[1, :a1 - a0] = lo1
                    thr_loc[2, :a1 - a0] = hi1
                    launches += 1
                del part_r, cand_r
            if world == 1:
                allt = thr_loc[None]
            else:
                allt = yield ("all_gather", thr_loc)                    # [world, nrow, per_r]
            rowthr = allt[:, 0].reshape(-1)[:n].contiguous()
            if one is not None:
                one["lo1"] = allt[:, 1].reshape(-1)[:n].contiguous()
                one["hi1"] = allt[:, 2].reshape(-1)[:n].contiguous()
            del Yc, ync, allt
            colthr = colb = None
            hi2_loc = torch.full((per,), float("inf"), dtype=torch.float32, device=dev) if one is not None else None
            if ns > 0:
                # column bounds: this rank's targets against a sample of the sources
                if pre is not None:
                    Xs = xns = part_s = None
                    cand_s = pre["cand_s"]
                else:
                    Xs, xns = X.index_select(0, sel), xn.index_select(0, sel)
                    part_s = be.eval_rowtopk(Ys, Xs, yns, xns, ns, m)
                    _, cand_s = be.topk_merge_mean(part_s, csls_k, want_nv=False, want_cand=True)
                    launches += 2
                colthr, colb = be.col_threshold(cand_s, csls_k, yns)
                launches += 1
                if one is not None:
                    one["lo2"], hi2_loc[:ns] = be.spec_bounds(cand_s, one["c_diag"][c0:c1].contiguous(), csls_k, one["shift"],
                                                              one["delta"])
                    launches += 1
                del part_s, cand_s, Xs, xns
            if one is not None:
                if world == 1:
                    hi2 = hi2_loc[:n]
                else:
                    allh = yield ("all_gather", hi2_loc)                # [world, per]
                    hi2 = allh.reshape(-1)[:n].contiguous()
                # relaxed rank constants (see EpiRankBand for R, R', C, C'): with nv1 - g = 2 c_ii - 1 - nv2_i (the CSLS
                # distance of the own pair) R_i depends on the pair's COLUMN mean only, C'_j on its ROW mean only
                slack = one["eps"] + 1e-6
                cd = one["c_diag"]
                one["rk_r"] = 0.25 * (2.0 * xn[:n] + 2.0 * cd - 2.0 - hi2) - slack
                one["rk_rp"] = 0.25 * ((2.0 * xn[:n] + one["lo1"]) - 1.0) - 1e-6
            if ns > 0:
                if one is not None:
                    one["rk_c"] = 0.25 * (2.0 * yns + one["lo2"]) - 1e-6
                    one["rk_cp"] = 0.25 * (2.0 * yns + 2.0 * cd[c0:c1] - 1.0 - one["hi1"][c0:c1]) - slack
                    key = (n, ns, csls_k, X.shape[1])
                    rk_cap = _ONE_PASS_CAP.get(key) or round_up(ONE_PASS_STREAM_PER_TARGET * ns // max(1, be.num_sms()) + 4096, 1024)
                    (part, pidx, stream, stream_row, stream_cnt, one["stream"], one["stream_row"], one["cnt"]) = be.eval_onepass(
                        X, Ys, xn, yns, n, ns, colthr, colb, cap, rowthr, one["rk_r"].contiguous(), one["rk_rp"].contiguous(),
                        one["rk_c"].contiguous(), one["rk_cp"].contiguous(), rk_cap, nrm2)
                    one["cap_key"], one["rk_cap"] = key, rk_cap
                else:
                    part, pidx, stream, stream_row, stream_cnt = be.eval_rowcoltopk(X, Ys, xn, yns, n, ns, colthr, colb, cap, rowthr,
                                                                                    nrm2)
                col_val, col_idx, overflow = be.col_cand_reduce(stream, stream_row, stream_cnt, ns, csls_k)
                col_bound = colthr                 # nothing below a target's threshold was ever streamed
                launches += 4
                if int(overflow.item()) != 0:      # a candidate stream filled up: redo the columns the classic way
                    col_val = col_idx = col_bound = None
                del stream, stream_row
        elif ns > 0:
            part, pidx = be.eval_rowtopk(X, Ys, xn, yns, n, ns, want_idx=True)
            launches += 1
        if part is None:
            part = torch.full((1, n, KT), float("-inf"), dtype=torch.float32, device=dev)
            pidx = torch.full((1, n, KT), -1, dtype=torch.int32, device=dev)
        _, cand, cidx = be.topk_merge_mean(part, csls_k, want_nv=False, part_idx=pidx)
        del part, pidx
        launches += 1
        if world > 1:
            cidx = torch.where(cidx >= 0, cidx + c0, cidx)             # shard-local columns -> pair ids
            allc = yield ("all_gather", cand)                          # [world, n, KT]
            alli = yield ("all_gather", cidx)
            _, cand, cidx = be.topk_merge_mean(allc.contiguous(), csls_k, want_nv=False, part_idx=alli.contiguous())
            launches += 1
        if world == 1:
            nv1 = be.topk_rescore(X, Y, xn, yn, cidx, cand, csls_k, n, "rows", **kw)
        else:
            # every rank holds the merged candidates of all sources; each re-scores its own slice of them
            per_r = (n + world - 1) // world
            a0, a1 = min(rank * per_r, n), min((rank + 1) * per_r, n)
            nv1_loc = torch.zeros((per_r,), dtype=torch.float32, device=dev)
            if a1 > a0:
                nv1_loc[:a1 - a0] = be.topk_rescore(X[a0:a1], Y, xn[a0:a1], yn, cidx[a0:a1].contiguous(),
                                                    cand[a0:a1].contiguous(), csls_k, n, "rows")
            allv1 = yield ("all_gather", nv1_loc)                      # [world, per_r]
            nv1 = allv1.reshape(-1)[:n].contiguous()
        launches += 1
        # sweep 1': column neighbourhoods — this rank's targets against every source
        # (skipped when the two-sweep path already collected them from the same pass over S)
        nv2_loc = torch.zeros((per,), dtype=torch.float32, device=dev)
        if ns > 0:
            if col_val is None:
                part2, pidx2 = be.eval_rowtopk(Ys, X, yns, xn, ns, n, want_idx=True)
                _, col_val, col_idx = be.topk_merge_mean(part2, csls_k, want_nv=False, part_idx=pidx2)
                del part2, pidx2
                launches += 2
            nv2_loc[:ns] = be.topk_rescore(Ys, X, yns, xn, col_idx, col_val, csls_k, n, "cols", outsider_bound=col_bound, **kw)
            launches += 1
        if world == 1:
            nv2 = nv2_loc[:n]
        else:
            allv = yield ("all_gather", nv2_loc)                       # [world, per]
            nv2 = allv.reshape(-1)[:n].contiguous()

    # ground-truth scores of all pairs (n dot products; replicated on every rank)
    g = be.pair_score(X, Y, n, xn, yn, nv1, nv2, use_csls)
    launches += 1

    # rank counters: settled on the streamed candidates of the one-pass sweep when it ran, else by sweep 2
    cnt_row = torch.zeros((n,), dtype=torch.int32, device=dev)
    cnt_col_loc = torch.zeros((per,), dtype=torch.int32, device=dev)
    t3v = t3i = None
    one_info = None
    if ns > 0:
        nv2s = nv2[c0:c1] if use_csls else None
        done = False
        if use_csls and one is not None and "stream" in one:
            done, one_info, nl = _one_pass_ranks(be, one, X, Ys, xn, yns, nv1, nv2s, g, c0, n, ns, cnt_row, cnt_col_loc)
            launches += nl
        if not done:
            t3v, t3i = be.eval_rank(X, Ys, xn, yns, nv1, nv2s, g, g[c0:c1], 0, c0, n, ns, use_csls, cnt_row, cnt_col_loc,
                                    want_top3, **kw)
            launches += 2                               # the sweep and the re-score of its deferred elements
    top3_idx = top3_val = None
    if want_top3:
        # each list holds the row's 4 nearest candidates (by the tensor-core score); merged here, exchanged when sharded,
        # then ordered by their canonical distances and cut to ret1..ret3
        if ns > 0:
            t3v, t3i = be.top4_merge(t3v, t3i)
            launches += 1
        else:
            t3v = torch.full((n, 4), float("-inf"), dtype=torch.float32, device=dev)
            t3i = torch.full((n, 4), 0x7FFFFFFF, dtype=torch.int32, device=dev)
    if world == 1:
        rank_l2r, rank_r2l = cnt_row, cnt_col_loc[:n]
    else:
        rank_l2r = yield ("all_reduce", cnt_row)
        allc = yield ("all_gather", cnt_col_loc)
        rank_r2l = allc.reshape(-1)[:n].contiguous()
        if want_top3:
            gv = yield ("all_gather", t3v.contiguous())                # [world, n, 4]
            gi = yield ("all_gather", t3i.contiguous())
            t3v, t3i = be.top4_merge(gv.contiguous(), gi.contiguous())
            launches += 1
    if want_top3:
        t3v, t3i = be.top3_rescore(X, Y, xn, yn, nv1, nv2, use_csls, t3i)
        launches += 1
        top3_idx, top3_val = t3i[:, :3], t3v[:, :3]
    return AlignRanks(rank_l2r, rank_r2l, nv1, nv2, g, top3_idx, top3_val, launches,
                      {"world": world, "rank": rank, "shard": (c0, c1), "rank_sweep": dict(getattr(be, "LAST_RANK_INFO", {})),
                       "neighbourhoods": dict(getattr(be, "LAST_TOPK_INFO", {})), "one_pass": one_info})


def _one_pass_ranks(be, one, X, Ys, xn, yns, nv1, nv2s, g, c0: int, n: int, ns: int, cnt_row, cnt_col_loc):
    """Rank counters from the streamed candidates of the one-pass sweep. Returns (done, info, launches); done False means
    the classic sweep 2 has to run (a stream overflowed, a guaranteed bound was violated, or too many guesses failed) —
    the counters are zero again in that case."""
    eps = one["eps"]
    gs = g[c0:c0 + ns]
    base_r = (2.0 * xn[:n] + nv1) - 1.0
    R, Rp = 0.25 * (base_r - g), 0.25 * base_r
    base_c = 2.0 * yns + nv2s
    C, Cp = 0.25 * base_c, 0.25 * (base_c - gs)
    tol = eps + 5e-7
    row_ok = one["rk_r"] <= R - tol
    col_ok = one["rk_cp"] <= Cp - tol
    broken = (one["rk_rp"] > Rp).sum() + (one["rk_c"] > C).sum()       # provable bounds: never expected
    overflow, deferred = be.rank_judge(X, Ys, xn, yns, nv1, nv2s, g, gs, 0, c0, one["stream"], one["stream_row"], one["cnt"],
                                       R.contiguous(), Rp.contiguous(), C.contiguous(), Cp.contiguous(),
                                       row_ok.to(torch.uint8), col_ok.to(torch.uint8), eps, cnt_row, cnt_col_loc)
    status = torch.stack([overflow[0].to(torch.int64), (~row_ok).sum(), (~col_ok).sum(), broken, one["cnt"].max().to(torch.int64),
                          one["cnt"].to(torch.int64).sum()]).tolist()
    ovf, fail_r, fail_c, brk, cnt_max, streamed = (int(v) for v in status)
    info = {"streamed": streamed, "deferred": deferred, "failed_rows": fail_r, "failed_cols": fail_c, "eps": eps,
            "stream_cap": one["rk_cap"], "stream_max": cnt_max, "fallback": None}
    launches = 2
    if ovf:
        _ONE_PASS_CAP[one["cap_key"]] = one["rk_cap"] * 4                # (the stream counters saturate) for the next evaluation
        info["fallback"] = "rank stream overflow"
    elif brk:
        info["fallback"] = "a lower bound from the sample exceeded the final neighbourhood mean"
    elif fail_r / n + fail_c / ns > ONE_PASS_RECOUNT_MAX_FRAC:
        info["fallback"] = "too many failed guesses"
    if info["fallback"] is not None:
        cnt_row.zero_()
        cnt_col_loc.zero_()
        return False, info, launches
    if cnt_max * 2 > one["rk_cap"]:
        _ONE_PASS_CAP[one["cap_key"]] = round_up(int(cnt_max * 2.5) + 4096, 1024)
    if fail_r:
        rows = (~row_ok).nonzero().reshape(-1).to(torch.int32)
        if fail_r <= ONE_PASS_EXHAUSTIVE_MAX:
            be.rank_exhaustive(X, Ys, xn, yns, nv1, nv2s, g, rows, 0, c0, True, False, cnt_row, ns)
        else:
            cnt_row[rows.long()] = be.rank_recount_rows(X, Ys, xn, yns, nv1, nv2s, g, gs, rows, 0, c0, ns, False, eps)
        launches += 2
    if fail_c:
        cols = (~col_ok).nonzero().reshape(-1).to(torch.int32)
        if fail_c <= ONE_PASS_EXHAUSTIVE_MAX:
            be.rank_exhaustive(Ys, X, yns, xn, nv2s, nv1, gs.contiguous(), cols, c0, 0, True, True, cnt_col_loc, n)
        else:
            cnt_col_loc[cols.long()] = be.rank_recount_rows(Ys, X, yns, xn, nv2s, nv1, gs.contiguous(), g, cols, c0, 0, n, True, eps)
        launches += 2
    return True, info, launches


def _drive_with_torch_distributed(gen, group):
    import torch.distributed as dist
    world = dist.get_world_size(group)
    try:
        req = next(gen)
        while True:
            op, t = req
            if op == "all_gather":
                flat = torch.empty((world * t.numel(),), dtype=t.dtype, device=t.device)
                dist.all_gather_into_tensor(flat, t.contiguous().reshape(-1), group=group)
                out = flat.view(world, *t.shape)
            elif op == "all_reduce":
                out = t.contiguous()
                dist.all_reduce(out, group=group)
            else:
                raise AssertionError(op)
            req = gen.send(out)
    except StopIteration as stop:
        return stop.value


def _world_rank(group) -> tuple[int, int]:
    if group is None:
        return 1, 0
    import torch.distributed as dist
    return dist.get_world_size(group), dist.get_rank(group)


def _run_steps(gen, group=None):
    """The result of an _align_ranks_steps generator: through torch.distributed with a group, else on this rank alone."""
    if group is not None:
        return _drive_with_torch_distributed(gen, group)
    try:
        next(gen)
    except StopIteration as stop:
        return stop.value
    raise AssertionError("single-rank evaluation requested a collective")


def _result(res: AlignRanks, launches: int, **extra) -> dict:
    """What the evaluate_alignment* entry points return: Hits@k / MR / MRR of both directions and the ranks."""
    return {"l2r": metrics_from_ranks(res.rank_l2r), "r2l": metrics_from_ranks(res.rank_r2l), "ranks": res,
            "launches": launches, **extra}


def simulate_sharded(make_gen, world: int):
    """Run `world` rank generators in lockstep inside one process (used by tests and single-GPU checks of the
    sharding logic): make_gen(rank) -> generator as produced by _align_ranks_steps."""
    gens = [make_gen(r) for r in range(world)]
    results = [None] * world
    reqs = []
    for r, gnr in enumerate(gens):
        try:
            reqs.append(next(gnr))
        except StopIteration as stop:
            results[r] = stop.value
            reqs.append(None)
    while any(q is not None for q in reqs):
        if any(q is None for q in reqs):
            raise AssertionError("ranks disagree on the number of collectives")
        op = reqs[0][0]
        if any(q[0] != op for q in reqs):
            raise AssertionError("ranks disagree on the collective sequence")
        if op == "all_gather":
            out = torch.stack([q[1] for q in reqs], 0)
            outs = [out.clone() for _ in range(world)]
        else:
            tot = reqs[0][1].clone()
            for q in reqs[1:]:
                tot += q[1]
            outs = [tot.clone() for _ in range(world)]
        nxt = []
        for r, gnr in enumerate(gens):
            try:
                nxt.append(gnr.send(outs[r]))
            except StopIteration as stop:
                results[r] = stop.value
                nxt.append(None)
        reqs = nxt
    return results


def _pending_status(res: AlignRanks, xn, yn, n: int) -> torch.Tensor:
    """int64 [4] on the device: (largest squared row norm in units of 1e-6, flagged rows, flagged columns, deferred)."""
    info = res.info
    nb = info["neighbourhoods"]
    z = torch.zeros((1,), dtype=torch.int64, device=xn.device)
    mx = (torch.maximum(xn[:n].max(), yn[:n].max()).double() * 1e6).to(torch.int64).reshape(1)
    fr = nb["rows"]["flagged_dev"].to(torch.int64) if "rows" in nb else z
    fc = nb["cols"]["flagged_dev"].to(torch.int64) if "cols" in nb else z
    df = info["rank_sweep"]["deferred_dev"].to(torch.int64) & 0xFFFFFFFF
    return torch.cat([mx, fr, fc, df])


def _resolve_pending(res: AlignRanks, status) -> bool:
    """Turn the device counters of a lazy evaluation into the usual info entries; False if an assumption failed (rows not
    unit norm, deferral list overflowed) and the result must not be used."""
    mx, fr, fc, df = (int(v) for v in status.tolist())
    nb, rs = res.info["neighbourhoods"], res.info["rank_sweep"]
    ok = mx <= int(LAZY_NORM2_BOUND * 1e6) and df <= rs["cap"]
    for tag, cnt in (("rows", fr), ("cols", fc)):
        if tag in nb:
            budget = nb[tag]["budget_rows"]
            nb[tag] = {"flagged": cnt, "unverified": max(0, cnt - budget)}
    rs.pop("deferred_dev", None)
    rs["deferred"] = df
    return ok


def _align_ranks_lazy(be, X, Y, xn, yn, n, csls_k, use_csls, want_top3):
    """Single-rank, three-sweep evaluation without any host synchronisation until ONE read of four counters at the end
    (what makes the evaluation of a reference-sized test set — 10 500 pairs, every epoch with --eval_epoch 1 — launch
    bound otherwise: ~8 round trips). Returns None when the read shows that an assumption did not hold."""
    res = _run_steps(_align_ranks_steps(be, X, Y, xn, yn, n, csls_k, use_csls, want_top3, 1, 0, False, lazy=True))
    status = _pending_status(res, xn, yn, n).cpu()        # the one synchronisation
    if not _resolve_pending(res, status):
        return None
    nb = res.info["neighbourhoods"]
    if any(v.get("unverified", 0) for v in nb.values()):
        import warnings
        warnings.warn("snag_b200: some CSLS neighbourhoods could not be verified within the exhaustive budget", RuntimeWarning)
    return res


def align_ranks(X: torch.Tensor, Y: torch.Tensor, xn: torch.Tensor, yn: torch.Tensor, n: int, csls_k: int = 10,
                use_csls: bool = True, want_top3: bool = False, group=None, _backend=None,
                two_sweep: bool = True, lazy: bool | None = None, one_pass: bool | None = None,
                pre: dict | None = None) -> AlignRanks:
    """Fused evaluation of n aligned pairs (x_i <-> y_i).

    X, Y : bf16 operands [>=n, Dpad] from ops.prep_bf16; xn, yn : their squared norms [n].
    With `group` (a torch.distributed process group, NCCL on GPUs) every rank holds all of X and Y and sweeps
    only its own shard of the targets.
    one_pass (default ONE_PASS; n >= TWO_SWEEP_MIN_N with CSLS and without the prediction file): rank verdicts are taken
    on candidates streamed out of the single main sweep instead of a second sweep (info["one_pass"] reports the volume,
    the guesses that failed and any fallback); the result is the same bit for bit."""
    if use_csls and not 1 <= csls_k <= KT:
        raise SnagError(f"csls_k={csls_k} unsupported: the fused CSLS path keeps {KT} candidates per row")
    if use_csls and csls_k > n:
        # torch.topk raises in the reference (src/utils.py:431) when k exceeds the matrix side
        raise ValueError(f"csls_k={csls_k} exceeds the number of evaluated pairs n={n}")
    # The s-space pre-filter margins inside the sweeps are derived for unit rows (what main.py:379's F.normalize
    # produces; the re-score tolerances scale with the norms, the in-kernel margins do not): refuse rows that are far
    # from that instead of silently weakening the guarantee. Squared norms up to 8 are let through for small exact
    # (dyadic) test inputs.
    be = _cuda_ops if _backend is None else _backend     # test seam: host-logic tests run the generator on a CPU stand-in
    world, rank = _world_rank(group)
    if lazy is None:
        lazy = world == 1 and _backend is None and n < TWO_SWEEP_MIN_N
    if lazy:
        res = _align_ranks_lazy(be, X, Y, xn, yn, n, csls_k, use_csls, want_top3)
        if res is not None:
            return res                                   # else: an assumption did not hold — take the synchronising path
    if float(torch.maximum(xn[:n].max(), yn[:n].max()).item()) > 8.0:
        raise SnagError("align_ranks expects L2-normalised rows (evaluate_alignment(normalize=True))")
    if pre is not None and (world != 1 or not use_csls or two_sweep_plan(n, csls_k) is None or not two_sweep):
        raise ValueError("pre-computed sample pre-passes apply to the single-rank two-sweep CSLS path only")
    return _run_steps(_align_ranks_steps(be, X, Y, xn, yn, n, csls_k, use_csls, want_top3, world, rank, two_sweep,
                                         one_pass=one_pass, pre=pre), group)


# =================================================================================================
# metrics (host glue; follows main.py:380-436 operation by operation)
# =================================================================================================
@dataclass
class AlignMetrics:
    acc: np.ndarray      # np.float32 [3]  Hits@1/10/50, rounded to 4 decimals like the reference
    mr: float            # mean rank, 1-based
    mrr: float
    hits: np.ndarray     # int64 [3] raw counts


def metrics_from_ranks(ranks, top_k=TOP_K) -> AlignMetrics:
    """Hits@k / MR / MRR from 0-based integer ranks, reproducing the reference's accumulators:
    hit counters are np.float32 (main.py:382-383), mean uses Python ints, mrr is a Python float summed in
    index order (main.py:403-404) -> np.cumsum in float64 is the same sequence of additions."""
    r = np.asarray(ranks.detach().cpu().numpy() if isinstance(ranks, torch.Tensor) else ranks)
    n = r.shape[0]
    if n == 0:
        raise ValueError("no test pairs")
    hits = np.array([np.count_nonzero(r < k) for k in top_k], dtype=np.int64)
    acc = np.zeros((len(top_k),), dtype=np.float32)
    for i in range(len(top_k)):
        acc[i] = round(np.float32(hits[i]) / n, 4)
    mr = float(int(r.sum(dtype=np.int64)) + n) / n                 # sum of the 1-based ranks, exact in integers
    # 1 / (rank + 1) in float64 (rank + 1 is exact), then the SEQUENTIAL left-to-right sum of main.py:404 — accumulate, not
    # np.sum, whose pairwise summation rounds differently. In place: one 8 MB buffer at 1M pairs (this runs on the host after
    # every evaluation; at 8 GPUs it is a visible part of the step).
    rec = r.astype(np.float64)
    rec += 1.0
    np.reciprocal(rec, out=rec)
    mrr = float(np.add.accumulate(rec, out=rec)[-1]) / n
    return AlignMetrics(acc, mr, mrr, hits)


class _GraphedEvaluation:
    """The whole single-GPU evaluation of a reference-sized test set (prologue, three sweeps, merges, canonical
    re-scores, rank sweep) captured ONCE in a CUDA graph for a fixed problem shape and replayed with a single launch.
    Possible because the lazy path never talks to the host and every entry point of libsnag_b200.so only enqueues on the
    stream it is given (TMA descriptors travel by value in the kernel parameters). Inputs are copied into static
    buffers before a replay; the outputs are cloned out of the graph's memory pool afterwards."""

    def __init__(self, emb_shape, n: int, csls: bool, csls_k: int, want_top3: bool, normalize: bool, device):
        self.emb = torch.zeros(emb_shape, dtype=torch.float32, device=device)
        self.left = torch.zeros((n,), dtype=torch.int64, device=device)
        self.right = torch.zeros((n,), dtype=torch.int64, device=device)
        self.n, self.args = n, (csls_k, csls, want_top3)
        self.normalize = normalize

        def run():
            X, xn = _cuda_ops.prep_bf16(self.emb, self.left, self.normalize)
            Y, yn = _cuda_ops.prep_bf16(self.emb, self.right, self.normalize)
            res = _run_steps(_align_ranks_steps(_cuda_ops, X, Y, xn, yn, n, csls_k, csls, want_top3, 1, 0, False, lazy=True))
            return res, _pending_status(res, xn, yn, n)

        self._run = run

    def capture(self, final_emb, test_left, test_right):
        self._load(final_emb, test_left, test_right)
        side = torch.cuda.Stream(device=self.emb.device)
        side.wait_stream(torch.cuda.current_stream(self.emb.device))
        with torch.cuda.stream(side):
            self._run()                                   # lazy initialisations (kernel attributes) outside the capture
        torch.cuda.current_stream(self.emb.device).wait_stream(side)
        torch.cuda.synchronize(self.emb.device)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.res, self.status = self._run()
        self.pending = {"neighbourhoods": {k: dict(v) for k, v in self.res.info["neighbourhoods"].items()},
                        "rank_sweep": dict(self.res.info["rank_sweep"])}

    def _load(self, final_emb, test_left, test_right):
        self.emb.copy_(final_emb)
        self.left.copy_(test_left)
        self.right.copy_(test_right)

    def __call__(self, final_emb, test_left, test_right):
        self._load(final_emb, test_left, test_right)
        self.graph.replay()
        status = self.status.cpu()                        # the one synchronisation
        r = self.res
        c = lambda t: None if t is None else t.clone()
        out = AlignRanks(c(r.rank_l2r), c(r.rank_r2l), c(r.nv1), c(r.nv2), c(r.g), c(r.top3_idx), c(r.top3_val), r.launches,
                         {**r.info, "neighbourhoods": {k: dict(v) for k, v in self.pending["neighbourhoods"].items()},
                          "rank_sweep": dict(self.pending["rank_sweep"]), "cuda_graph": True})
        return out if _resolve_pending(out, status) else None


_GRAPHS: dict = {}
USE_EVAL_GRAPH = True       # evaluate_alignment replays a CUDA graph for single-GPU problems below TWO_SWEEP_MIN_N pairs


def _graphed(final_emb, test_left, test_right, csls, csls_k, want_top3, normalize):
    """AlignRanks through a cached CUDA graph, or None (capture unavailable / an assumption of the lazy path failed)."""
    n = test_left.numel()
    key = (tuple(final_emb.shape), n, bool(csls), int(csls_k), bool(want_top3), bool(normalize), final_emb.device.index)
    g = _GRAPHS.get(key)
    if g is False:
        return None
    if g is None:
        if len(_GRAPHS) >= 8:
            _GRAPHS.clear()
        try:
            g = _GraphedEvaluation(tuple(final_emb.shape), n, csls, csls_k, want_top3, normalize, final_emb.device)
            g.capture(final_emb, test_left, test_right)
        except Exception:                    # noqa: BLE001 — e.g. a capture already in progress on this stream: run eagerly
            _GRAPHS[key] = False
            return None
        _GRAPHS[key] = g
    return g(final_emb, test_left, test_right)


PRECISIONS = ("bf16", "fp32")
EVAL_PRECISION = "bf16"     # what Runner._test evaluates with (python -m snag_b200.patch --eval-precision fp32 sets it)


def _check_precision(precision: str) -> None:
    if precision not in PRECISIONS:
        raise ValueError(f"precision={precision!r}: expected one of {PRECISIONS}")


def _check_eval_args(what: str, final_emb, test_left, test_right, csls: bool, csls_k: int) -> int:
    """The refusals evaluate_alignment and evaluate_alignment_l1 share; returns the number of pairs n."""
    n = test_left.numel()
    if test_right.numel() != n:
        raise ValueError("test_left and test_right must pair up")
    if csls and csls_k < 1:
        raise ValueError(f"csls_k={csls_k}")
    if csls and csls_k > n:
        raise ValueError(f"csls_k={csls_k} exceeds the number of evaluated pairs n={n}")
    if not final_emb.is_cuda:
        raise SnagError(f"{what}: final_emb must live on the GPU (there is no CPU path)")
    return n


def evaluate_alignment(final_emb: torch.Tensor, test_left: torch.Tensor, test_right: torch.Tensor, csls: bool = True,
                       csls_k: int = 10, want_top3: bool = False, normalize: bool = True, group=None,
                       graph: bool | None = None, precision: str = "bf16") -> dict:
    """The evaluation a user of the reference gets from Runner._test, as a function:
    final_emb [N, D] fp32 (device), test_left/right LongTensor [n] -> metrics for both directions.
    graph (default: on for a single GPU and fewer than TWO_SWEEP_MIN_N pairs): replay the evaluation as one CUDA graph
    captured on the first call with this shape — the reference evaluates the same test set after every epoch.
    precision: "bf16" (default) ranks the normalised rows rounded to bf16; "fp32" ranks the unrounded fp32 rows, as the
    reference does (snag_b200.fp32: split-bf16 sweeps, canonical re-scores on the fp32 rows), so that ranks, nv1 / nv2,
    g and Hits@k / MR / MRR equal the reference's bit for bit. fp32 needs csls_k <= KT and runs without the CUDA graph."""
    _check_precision(precision)
    if precision == "fp32" and csls and csls_k > KT:
        raise SnagError(f"precision='fp32' with csls_k={csls_k} > {KT}: the materialised evaluation is bf16 only")
    n = _check_eval_args("evaluate_alignment", final_emb, test_left, test_right, csls, csls_k)
    if precision == "fp32":
        return _evaluate_fp32(final_emb, test_left, test_right, csls, csls_k, want_top3, normalize, group)
    if csls and csls_k > KT:
        # the fused sweeps keep KT candidates per entity; larger neighbourhoods (the reference takes any k) are evaluated
        # on the materialised matrix
        return evaluate_alignment_materialised(final_emb, test_left, test_right, csls, csls_k, want_top3, normalize, group)
    if graph is None:
        graph = USE_EVAL_GRAPH and group is None and n < TWO_SWEEP_MIN_N and not torch.cuda.is_current_stream_capturing()
    if graph and group is None and final_emb.is_cuda and final_emb.dtype == torch.float32:
        res = _graphed(final_emb.contiguous(), test_left.to(torch.int64), test_right.to(torch.int64), csls, csls_k,
                       want_top3, normalize)
        if res is not None:
            return _result(res, res.launches + 2)
    X, xn = _cuda_ops.prep_bf16(final_emb, test_left.to(torch.int64).contiguous(), normalize)
    Y, yn = _cuda_ops.prep_bf16(final_emb, test_right.to(torch.int64).contiguous(), normalize)
    res = align_ranks(X, Y, xn, yn, n, csls_k, csls, want_top3, group)
    return _result(res, res.launches + 2)


def _evaluate_fp32(final_emb, test_left, test_right, csls: bool, csls_k: int, want_top3: bool, normalize: bool, group) -> dict:
    """evaluate_alignment(precision="fp32"): the fused evaluation with the kernel backend snag_b200.fp32."""
    from . import fp32
    n = test_left.numel()
    X, xn = fp32.prep(final_emb, test_left.to(torch.int64).contiguous(), normalize, 0)
    Y, yn = fp32.prep(final_emb, test_right.to(torch.int64).contiguous(), normalize, 1)
    if float(torch.maximum(xn[:n].max(), yn[:n].max()).item()) > 8.0:
        raise SnagError("the fused evaluation expects L2-normalised rows (evaluate_alignment(normalize=True))")
    res = _run_steps(_align_ranks_steps(fp32, X, Y, xn, yn, n, csls_k, csls, want_top3, *_world_rank(group)), group)
    res.info["precision"] = "fp32"
    return _result(res, res.launches + 4)


def evaluate_alignment_materialised(final_emb: torch.Tensor, test_left: torch.Tensor, test_right: torch.Tensor, csls: bool = True,
                                    csls_k: int = 10, want_top3: bool = False, normalize: bool = True, group=None) -> dict:
    """Runner._test (main.py:379-429) for CSLS neighbourhoods larger than the fused path's KT candidates (csls_k up to
    ops.CSLS_MATRIX_K_MAX; no script of the reference goes beyond 10): the reference's own composition —
    pairwise_distances -> 1 - csls_sim(1 - d, k) -> rank of the diagonal — with the [n, n] fp32 matrix materialised on
    the device by the drop-in kernels (tensor-core distances, radix-select neighbourhood means, counting ranks with the
    stable-sort tie-break). Single GPU; needs 3 * 4 n^2 bytes."""
    if group is not None:
        raise SnagError(f"csls_k={csls_k} > {KT}: the materialised evaluation is not sharded")
    n = test_left.numel()

    def distances():
        X, xn = _cuda_ops.prep_bf16(final_emb, test_left.to(torch.int64).contiguous(), normalize)
        Y, yn = _cuda_ops.prep_bf16(final_emb, test_right.to(torch.int64).contiguous(), normalize)
        return _cuda_ops.sim_write(X, Y, xn, yn, n, n, mode=1)                       # main.py:386

    return _materialised(distances, n, final_emb.device, csls, csls_k, want_top3,
                         {"materialised": True, "csls_k": int(csls_k)})


def _materialised(distances, n: int, device, csls: bool, csls_k: int, want_top3: bool, info: dict) -> dict:
    """The reference's composition on the materialised [n, n] fp32 matrix that distances() builds: csls_sim on
    1 - distance, counting ranks of the diagonal with the stable-sort tie-break, and the top 3 of a stable sort."""
    free, _total = torch.cuda.mem_get_info(device)
    if 3 * 4 * n * n > free:
        raise SnagError(f"csls_k={csls_k} > {KT} needs the materialised {n} x {n} matrix, which does not fit this device")
    dist = distances()
    nv1 = nv2 = None
    if csls:
        out, nv1, nv2 = _cuda_ops.csls_sim_matrix(1 - dist, int(csls_k))              # main.py:393
        dist = 1 - out
        del out
    rank_l2r, rank_r2l = _cuda_ops.matrix_rank(dist)
    top3_idx = top3_val = None
    if want_top3:
        order = torch.sort(dist, dim=1, stable=True)
        top3_idx, top3_val = order[1][:, :3].to(torch.int32), order[0][:, :3]
    return _result(AlignRanks(rank_l2r, rank_r2l, nv1, nv2, torch.diagonal(dist).clone(), top3_idx, top3_val, 7, info), 7)


def evaluate_alignment_l1(final_emb: torch.Tensor, test_left: torch.Tensor, test_right: torch.Tensor, csls: bool = True,
                          csls_k: int = 10, want_top3: bool = False, group=None) -> dict:
    """Runner._test with --distance 1 (main.py:379, 387-429). The reference normalises on the device, moves both sides
    to the host and calls scipy's cdist(metric="cityblock"). Here the rows are normalised and gathered in torch (the same
    operands), and the evaluation is the fused one of evaluate_alignment with the L1 kernels of snag_b200.l1: a CUDA-core
    sweep in fp32 whose verdicts inside its error bound are re-judged with the canonical arithmetic (fp64 index-order
    sums rounded once, the reference's fp32 CSLS chain), so ranks, nv1 / nv2, g and the prediction ids equal the
    reference's without the [n, n] matrix. With `group` every rank passes the same final_emb, sweeps its own shard of the
    targets and gets the full metrics. CSLS neighbourhoods larger than the KT candidates of the fused sweep are evaluated
    on the materialised matrix (single GPU)."""
    materialised = csls and not 1 <= csls_k <= KT
    if materialised and group is not None:
        raise SnagError(f"csls_k={csls_k} > {KT}: the materialised evaluation is not sharded")
    n = _check_eval_args("evaluate_alignment_l1", final_emb, test_left, test_right, csls, csls_k)
    fe = torch.nn.functional.normalize(final_emb.float())                       # main.py:379
    left, right = test_left.to(torch.int64), test_right.to(torch.int64)
    if materialised:            # fp64 index-order L1 sums
        return _materialised(lambda: _cuda_ops.l1_distance(fe.index_select(0, left).contiguous(),
                                                             fe.index_select(0, right).contiguous()),
                             n, fe.device, True, csls_k, want_top3, {"distance": 1, "materialised": True})
    from . import l1
    X, xn = l1.prep(fe, left)
    Y, yn = l1.prep(fe, right)
    res = _run_steps(_align_ranks_steps(l1, X, Y, xn, yn, n, csls_k, csls, want_top3, *_world_rank(group), two_sweep=False),
                     group)
    res.info["distance"] = 1
    return _result(res, res.launches + 2)


STREAM_CHUNK_ROWS = 65536      # rows per host -> device chunk of the streamed entry point (315 MB at D = 1200: ~6 ms of PCIe 5)
_PINNED: dict = {}


def _pinned(shape, key):
    """A cached pinned staging buffer (pinning 150 MB costs more than the copy it speeds up)."""
    buf = _PINNED.get(key)
    if buf is None or tuple(buf.shape) != tuple(shape):
        if len(_PINNED) > 4:
            _PINNED.clear()
        buf = torch.empty(shape, dtype=torch.float32).pin_memory()
        _PINNED[key] = buf
    return buf


def _stream_in_with_prepasses(src_rows, tgt_rows, n: int, csls_k: int, normalize: bool, device, m: int, timeline: dict | None = None):
    """Host -> device transfer of both tables in row chunks on a copy stream, overlapped with everything that needs only
    the rows that have arrived: normalise + round (prep_bf16) and the two sample pre-passes of the two-sweep evaluation.
    Order: a few source chunks, the m sampled TARGET rows (gathered on the host into pinned staging while those chunks
    are in flight), the remaining sources — each chunk's row pre-pass (its sources x the sampled targets) runs as soon
    as it lands — then the targets, each chunk's column pre-pass running against the sampled sources, which are on the
    device by then. Returns X, Y, xn, yn and the merged pre-pass candidates for align_ranks(pre=...). The PCIe copy
    (9.6 GB at 1M x 1200) is the critical path; 2 x m/n of a sweep and the prologue hide behind it."""
    be = _cuda_ops
    d = src_rows.shape[1]
    dpad = round_up(d, 64)
    cur = torch.cuda.current_stream(device)
    copy_s = torch.cuda.Stream(device=device)
    copy_s.wait_stream(cur)
    sel, selc = _sample_rows(n, m, device)
    xs = torch.empty((n, d), dtype=torch.float32, device=device)
    ys = torch.empty((n, d), dtype=torch.float32, device=device)
    X = torch.empty((n, dpad), dtype=torch.bfloat16, device=device)
    Y = torch.empty((n, dpad), dtype=torch.bfloat16, device=device)
    xn = torch.empty((n,), dtype=torch.float32, device=device)
    yn = torch.empty((n,), dtype=torch.float32, device=device)
    cand_r = torch.empty((n, KT), dtype=torch.float32, device=device)
    cand_s = torch.empty((n, KT), dtype=torch.float32, device=device)
    ysamp = torch.empty((m, d), dtype=torch.float32, device=device)
    bounds = [(r0, min(n, r0 + STREAM_CHUNK_ROWS)) for r0 in range(0, n, STREAM_CHUNK_ROWS)]
    events = {}
    lead = min(3, len(bounds))     # source chunks queued ahead of the sampled rows: the DMA engine stays busy during the host gather

    def queue(tag, host, dst, chunks):
        with torch.cuda.stream(copy_s):
            for i in chunks:
                r0, r1 = bounds[i]
                dst[r0:r1].copy_(host[r0:r1], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_s)
                events[tag, i] = ev

    # ONE copy stream, in the order the data is needed (copies queued on a second stream were measured to be served only
    # after the first stream's queue had drained): a few source chunks, the sampled target rows — gathered on the host
    # into pinned staging while those chunks are in flight — the remaining sources, then the targets
    queue("x", src_rows, xs, range(lead))
    stage = _pinned((m, d), ("ysamp", m, d))
    torch.index_select(tgt_rows, 0, _sample_rows_host(n, m, device)[1], out=stage)
    with torch.cuda.stream(copy_s):
        ysamp.copy_(stage, non_blocking=True)
        ev_samp = torch.cuda.Event()
        ev_samp.record(copy_s)
    queue("x", src_rows, xs, range(lead, len(bounds)))
    queue("y", tgt_rows, ys, range(len(bounds)))

    def mark(name, stream):
        if timeline is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(stream)
            timeline[name] = ev

    mark("copies_done", copy_s)
    mark("start", cur)
    cur.wait_event(ev_samp)
    mark("sample_landed", cur)
    Yc, ync = be.prep_bf16(ysamp, None, normalize)
    launches = 1
    for i, (r0, r1) in enumerate(bounds):                           # sources: prologue + row pre-pass per chunk
        cur.wait_event(events["x", i])
        _, a = be.prep_bf16(xs[r0:r1], None, normalize, out=X[r0:r1])
        xn[r0:r1] = a
        part = be.eval_rowtopk(X[r0:r1], Yc, xn[r0:r1], ync, r1 - r0, m)
        _, c = be.topk_merge_mean(part, csls_k, want_nv=False, want_cand=True)
        cand_r[r0:r1] = c
        launches += 3
    mark("sources_done", cur)
    Xs, xns = X.index_select(0, sel), xn.index_select(0, sel)
    for i, (r0, r1) in enumerate(bounds):                           # targets: prologue + column pre-pass per chunk
        cur.wait_event(events["y", i])
        _, b = be.prep_bf16(ys[r0:r1], None, normalize, out=Y[r0:r1])
        yn[r0:r1] = b
        part = be.eval_rowtopk(Y[r0:r1], Xs, yn[r0:r1], xns, r1 - r0, m)
        _, c = be.topk_merge_mean(part, csls_k, want_nv=False, want_cand=True)
        cand_s[r0:r1] = c
        launches += 3
    mark("targets_done", cur)
    # every copy has been waited for on the current stream: the staging buffers may be reused by later allocations on it
    return X, Y, xn, yn, {"cand_r": cand_r, "cand_s": cand_s}, launches


def evaluate_alignment_host(src_rows: torch.Tensor, tgt_rows: torch.Tensor, n: int, row0: int = 0, csls: bool = True,
                            csls_k: int = 10, normalize: bool = True, group=None, device=None, stream_in: bool | None = None,
                            precision: str = "bf16") -> dict:
    """End-to-end entry point from HOST memory: `src_rows` / `tgt_rows` are (ideally pinned) fp32 [m, D] host tensors
    holding pairs row0 .. row0+m of the n evaluated pairs — all of them on a single GPU, or this rank's contiguous
    slice (ceil(n / world) pairs per rank) when `group` is given. Copies them to the device, normalises and rounds
    them, exchanges the bf16 operands over NCCL so that every rank holds both tables, runs the sharded fused
    evaluation, brings the ranks back and reduces them to Hits@k / MR / MRR on the host.
    stream_in (default: single GPU, CSLS, n >= TWO_SWEEP_MIN_N): transfer the tables in chunks and run the prologue and
    the sample pre-passes on the chunks as they arrive (_stream_in_with_prepasses); the result is bit-identical.
    precision: "bf16" only (the fp32 evaluation takes device tables: evaluate_alignment(precision="fp32"))."""
    _check_precision(precision)
    if precision != "bf16":
        raise SnagError("evaluate_alignment_host evaluates bf16 operands only: use evaluate_alignment(precision='fp32')")
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device())
    m, d = src_rows.shape
    if tgt_rows.shape != (m, d):
        raise ValueError("source and target slices must have the same shape")
    if group is None:
        world, per = 1, n
        if m != n or row0 != 0:
            raise ValueError("without a process group the host buffers must hold all n pairs")
    else:
        import torch.distributed as dist
        world = dist.get_world_size(group)
        per = (n + world - 1) // world
        if row0 != dist.get_rank(group) * per or m != max(0, min(n, row0 + per) - row0):
            raise ValueError("host slice does not match this rank's share of the pairs")
    plan2 = two_sweep_plan(n, csls_k) if (csls and 1 <= csls_k <= KT and csls_k <= n) else None
    if stream_in is None:
        stream_in = world == 1 and plan2 is not None
    if stream_in:
        if world != 1 or plan2 is None:
            raise ValueError("stream_in applies to the single-GPU two-sweep CSLS evaluation (n >= TWO_SWEEP_MIN_N)")
        X, Y, xn, yn, pre, launches = _stream_in_with_prepasses(src_rows, tgt_rows, n, csls_k, normalize, device, plan2[0])
        res = align_ranks(X, Y, xn, yn, n, csls_k, csls, False, None, pre=pre)
        return _result(res, res.launches + launches, streamed=True)
    xs = src_rows.to(device, non_blocking=True)
    ys = tgt_rows.to(device, non_blocking=True)
    dpad = round_up(d, 64)
    Xl = torch.zeros((per, dpad), dtype=torch.bfloat16, device=device) if m < per else \
        torch.empty((per, dpad), dtype=torch.bfloat16, device=device)
    Yl = torch.zeros_like(Xl) if m < per else torch.empty_like(Xl)
    xnl = torch.zeros((per,), dtype=torch.float32, device=device)
    ynl = torch.zeros((per,), dtype=torch.float32, device=device)
    if m > 0:
        _, a = _cuda_ops.prep_bf16(xs, None, normalize, out=Xl)
        _, b = _cuda_ops.prep_bf16(ys, None, normalize, out=Yl)
        xnl[:m] = a
        ynl[:m] = b
    launches = 2
    if world == 1:
        X, Y, xn, yn = Xl, Yl, xnl, ynl
    else:
        X = torch.empty((world * per, dpad), dtype=torch.bfloat16, device=device)
        Y = torch.empty_like(X)
        xn = torch.empty((world * per,), dtype=torch.float32, device=device)
        yn = torch.empty_like(xn)
        dist.all_gather_into_tensor(X, Xl, group=group)
        dist.all_gather_into_tensor(Y, Yl, group=group)
        dist.all_gather_into_tensor(xn, xnl, group=group)
        dist.all_gather_into_tensor(yn, ynl, group=group)
    res = align_ranks(X, Y, xn[:n].contiguous(), yn[:n].contiguous(), n, csls_k, csls, False, group)
    return _result(res, res.launches + launches)


# =================================================================================================
# materialising drop-ins
# =================================================================================================
def pairwise_distances(x: torch.Tensor, y: torch.Tensor | None = None) -> torch.Tensor:
    """Drop-in for src/utils.py:202-218: dist[i,j] = clamp(||x_i||^2 + ||y_j||^2 - 2 x_i.y_j, 0), fp32 [n1,n2].
    Operands are rounded to bf16 for the tensor-core contraction; norms are those of the rounded rows."""
    x = x.contiguous().float()
    X, xn = _cuda_ops.prep_bf16(x, None, normalize=False)
    if y is None:
        Y, yn = X, xn
        n2 = x.shape[0]
    else:
        y = y.contiguous().float()
        Y, yn = _cuda_ops.prep_bf16(y, None, normalize=False)
        n2 = y.shape[0]
    return _cuda_ops.sim_write(X, Y, xn, yn, x.shape[0], n2, mode=1)


def csls_sim(sim_mat: torch.Tensor, k: int) -> torch.Tensor:
    """Drop-in for src/utils.py:417-435 on a materialised similarity matrix: 2*sim - mean(topk rows) - mean(topk cols).
    Bit-exact against the oracle for the same input (top-k selection, largest-first fp32 mean, two fp32 ops)."""
    out, _, _ = _cuda_ops.csls_sim_matrix(sim_mat.contiguous().float(), int(k))
    return out
