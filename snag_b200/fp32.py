"""Kernel backend of the fp32 evaluation (evaluate.evaluate_alignment(precision="fp32")): the entry points
evaluate._align_ranks_steps calls, over the UNROUNDED fp32 normalised rows.

Every table is carried as a SplitOperand: its fp32 rows [n, Dpad] (what the canonical re-scores read, through the
snag_*_f32 entry points) and a three-term bf16 split of them [n, 3 Dpad] (what the existing tcgen05 sweeps of
snag_b200.ops contract, unchanged): h = bf16(x), m = bf16(x - h), laid out [m | h | h] for sources and [h | m | h] for
targets, so that a sweep forms m_x h_y + h_x m_y + h_x h_y whichever operand comes first. The small terms come first:
the accumulator stays small for the first 2 Dpad k-steps. The candidate-list plumbing in score space (merges, bounds,
column reductions, the one-pass judge's counting) is shared with ops unchanged; only the error model differs:

    |s_tc - s_canonical| <= E_tc(Dpad) + 3 * 2^-16 * sum_k |x_k y_k| + 1/2 ulp_32(s)

E_tc is the tensor core's accumulation error on the split operands, measured (FP32_TC_DOT_ERR_PER_K); the split term
is proven (|x - h - m| <= 2^-16 |x|, and the dropped m_x m_y <= 2^-16 |x y|); subnormal m that the tensor cores may
flush add at most D * 2^-126 and are neglected. sum_k |x_k y_k| <= ||x|| ||y||."""
from __future__ import annotations

import torch

from . import ops
from ._lib import SnagError, call, current_stream, ptr
from .ops import (HALF_PREFILTER_NORM2_MAX, _need, col_cand_reduce, col_threshold, num_sms, round_up,  # noqa: F401
                  spec_bounds, top4_merge, topk_merge_mean)

LAST_TOPK_INFO: dict = {}
LAST_RANK_INFO: dict = {}

# E_tc: worst |s_tc - (exact m_x h_y + h_x m_y + h_x h_y)| of the split operands, measured on a B200 over 2 x 1.07e9
# adversarial pairs of unit rows (tests/test_fp32_eval_gpu.py::test_split_tensor_core_error_on_1e9_pairs): 9.45e-6 at
# Dpad = 1216 and 1.30e-5 at Dpad = 1856, i.e. 7.8e-9 and 7.0e-9 per element of Dpad (the small terms first keep it at
# the bf16 path's level, ops.TC_DOT_ERR_PER_K); bounded here by 9e-9, and the margins keep 4x over it. The whole error
# against the fp64 dot of the fp32 rows was 1.89e-5 / 2.17e-5 there.
FP32_TC_DOT_ERR_PER_K = 9e-9
SPLIT_REL_ERR = 3.0 * 2.0 ** -16        # proven: |x.y - (m_x h_y + h_x m_y + h_x h_y)| <= this * sum |x_k y_k|
HALF_ULP = 2.0 ** -24                   # half an fp32 ulp of the rounded canonical s (|s| < 2), per unit of ||x|| ||y||
RANK_BAND_MAX_CAP = 1 << 28


class SplitOperand:
    """A table of the fp32 evaluation: `split` bf16 [n, 3 Dpad] (sweep operand), `rows` fp32 [n, Dpad] (canonical
    re-scores), row for row. Supports what the evaluation driver does with its operands: .device, .shape (that of the
    fp32 rows), slicing of rows and index_select(0, ids)."""

    __slots__ = ("split", "rows")

    def __init__(self, split: torch.Tensor, rows: torch.Tensor):
        if split.shape[0] != rows.shape[0] or split.shape[1] != 3 * rows.shape[1]:
            raise ValueError("split must be [n, 3 Dpad] for rows [n, Dpad]")
        self.split, self.rows = split, rows

    @property
    def device(self):
        return self.rows.device

    @property
    def shape(self):
        return self.rows.shape

    def __getitem__(self, sl):
        return SplitOperand(self.split[sl], self.rows[sl])

    def index_select(self, dim: int, index: torch.Tensor) -> "SplitOperand":
        if dim != 0:
            raise ValueError("operands are gathered by rows")
        return SplitOperand(self.split.index_select(0, index), self.rows.index_select(0, index))


def prep(emb: torch.Tensor, idx: torch.Tensor | None, normalize: bool, side: int) -> tuple[SplitOperand, torch.Tensor]:
    """(gather ->) L2-normalise with prep_bf16's arithmetic, without rounding: the split operand of `side` (0 = sources,
    1 = targets) and ||row||^2 of the fp32 rows (fp64, index order, rounded once). snag_prep_split."""
    _need(emb, torch.float32, "emb", 2)
    if idx is not None:
        _need(idx, torch.int64, "idx", 1)
    n = emb.shape[0] if idx is None else idx.numel()
    if n == 0:
        raise ValueError("empty operand")
    d = emb.shape[1]
    dpad = round_up(d, 64)
    rows = torch.empty((n, dpad), dtype=torch.float32, device=emb.device)
    split = torch.empty((n, 3 * dpad), dtype=torch.bfloat16, device=emb.device)
    norm2 = torch.empty((n,), dtype=torch.float32, device=emb.device)
    call("snag_prep_split", ptr(emb), emb.stride(0), ptr(idx), n, d, int(normalize), int(side), ptr(rows), ptr(split), dpad,
         ptr(norm2), current_stream())
    return SplitOperand(split, rows), norm2


def _rows(t: SplitOperand, name: str) -> torch.Tensor:
    if not isinstance(t, SplitOperand):
        raise TypeError(f"{name} must be a fp32.SplitOperand (use fp32.prep)")
    _need(t.rows, torch.float32, name, 2)
    if t.rows.shape[1] % 64 or t.rows.data_ptr() % 16:
        raise ValueError(f"{name}: rows must be [n, multiple of 64] and 16-byte aligned")
    return t.rows


# ------------------------------------------------------------------------------------------------ error model
def tc_margin(dpad: int, norm: float = 1.0) -> float:
    """Half-width (in s) inside which a tensor-core verdict on split operands is not trusted, for fp32 rows of width dpad
    with ||x|| ||y|| <= norm: 4 x the measured accumulation bound, the proven split term, half an fp32 ulp of the
    canonical s, and 1e-6 for the roundings of the reference's fp32 chain and of the thresholds (as ops.tc_margin)."""
    nrm = max(1.0, norm)
    return max(ops.TC_MARGIN_FLOOR, 4.0 * FP32_TC_DOT_ERR_PER_K * dpad * nrm + (SPLIT_REL_ERR + HALF_ULP) * nrm + 1e-6)


def _error_scale(xn: torch.Tensor, yn: torch.Tensor, dpad: int) -> float:
    return tc_margin(dpad, float(torch.sqrt(xn.max() * yn.max()).item()))


def rank_band_eps(xn: torch.Tensor, yn: torch.Tensor, dpad: int) -> float:
    """Half-width of the rank sweep's deferral band (in s) for these fp32 rows."""
    return ops.RANK_BAND_EPS * _error_scale(xn, yn, dpad)


# ------------------------------------------------------------------------------------------------ sweeps (split operands)
def eval_rowtopk(X, Y, xn, yn, n1: int, n2: int, want_idx: bool = False):
    return ops.eval_rowtopk(X.split, Y.split, xn, yn, n1, n2, want_idx)


def eval_rowcoltopk(X, Y, xn, yn, n1: int, n2: int, colthr, colb, cta_cap: int, rowthr=None, norm2_max=None):
    return ops.eval_rowcoltopk(X.split, Y.split, xn, yn, n1, n2, colthr, colb, cta_cap, rowthr, norm2_max)


def eval_onepass(X, Y, xn, yn, n1: int, n2: int, colthr, colb, cta_cap: int, rowthr, rk_r, rk_rp, rk_c, rk_cp, rk_cap: int,
                 norm2_max=None):
    return ops.eval_onepass(X.split, Y.split, xn, yn, n1, n2, colthr, colb, cta_cap, rowthr, rk_r, rk_rp, rk_c, rk_cp, rk_cap,
                            norm2_max)


# ------------------------------------------------------------------------------------------------ canonical (fp32 rows)
def topk_rescore(A, B, an, bn, cand_idx, cand_val, k: int, n_b: int, tag: str = "rows", outsider_bound=None):
    """ops.topk_rescore on the fp32 rows: canonical neighbourhood means from the candidates, verified against the fp32
    error model; unverifiable rows are completed by an exhaustive canonical scan (or reported as unverified beyond
    ops.TOPK_EXHAUSTIVE_BUDGET)."""
    Ar, Br = _rows(A, "A"), _rows(B, "B")
    _need(cand_idx, torch.int32, "cand_idx", 2)
    _need(cand_val, torch.float32, "cand_val", 2)
    if outsider_bound is not None:
        _need(outsider_bound, torch.float32, "outsider_bound", 1)
    n_rows, dpad = cand_idx.shape[0], Ar.shape[1]
    dev, st = Ar.device, current_stream()
    nv = torch.empty((n_rows,), dtype=torch.float32, device=dev)
    flagged = torch.empty((n_rows,), dtype=torch.int32, device=dev)
    fcnt = torch.zeros((1,), dtype=torch.int32, device=dev)
    margin = _error_scale(an, bn, dpad)
    call("snag_topk_rescore_f32", ptr(Ar), ptr(Br), dpad, n_rows, ptr(an), ptr(bn), ptr(cand_idx), ptr(cand_val), k,
         ops.TOPK_VERIFY_DELTA * margin, ptr(outsider_bound), ptr(nv), ptr(flagged), ptr(fcnt), n_rows, None, None, st)
    n_flag = int(fcnt.item())
    info = {"flagged": n_flag, "unverified": 0}
    if n_flag:
        if float(n_flag) * n_b * dpad <= ops.TOPK_EXHAUSTIVE_BUDGET:
            call("snag_topk_exhaustive_f32", ptr(Ar), ptr(Br), dpad, n_b, ptr(an), ptr(bn), ptr(flagged), ptr(fcnt), n_rows, k,
                 ptr(nv), None, None, st)
        else:
            info["unverified"] = n_flag
            import warnings
            warnings.warn(f"snag_b200: {n_flag} {tag} neighbourhoods could not be verified against the canonical arithmetic "
                          f"within the exhaustive budget", RuntimeWarning, stacklevel=2)
    LAST_TOPK_INFO[tag] = info
    return nv


def pair_score(X, Y, n: int, xn, yn, nv1, nv2, use_csls: bool):
    Xr, Yr = _rows(X, "X"), _rows(Y, "Y")
    g = torch.empty((n,), dtype=torch.float32, device=Xr.device)
    call("snag_pair_score_f32", ptr(Xr), ptr(Yr), Xr.shape[1], n, ptr(xn), ptr(yn), ptr(nv1), ptr(nv2), int(use_csls), ptr(g),
         None, current_stream())
    return g


def pairs_dot(X, Y, rows: torch.Tensor, cols: torch.Tensor) -> torch.Tensor:
    """Canonical dot products of listed pairs of fp32 rows (X, Y: SplitOperand or fp32 [n, Dpad] tensors)."""
    Xr = X.rows if isinstance(X, SplitOperand) else X
    Yr = Y.rows if isinstance(Y, SplitOperand) else Y
    _need(Xr, torch.float32, "X", 2)
    _need(Yr, torch.float32, "Y", 2)
    _need(rows, torch.int32, "rows", 1)
    _need(cols, torch.int32, "cols", 1)
    if rows.numel() != cols.numel():
        raise ValueError("rows and cols must pair up")
    out = torch.empty((rows.numel(),), dtype=torch.float32, device=Xr.device)
    if rows.numel():
        call("snag_pairs_dot_f32", ptr(Xr), ptr(Yr), Xr.shape[1], ptr(rows), ptr(cols), rows.numel(), ptr(out), current_stream())
    return out


def eval_rank(X, Y, xn, yn, nv1, nv2, g_row, g_col, row_gid0: int, col_gid0: int, n1: int, n2: int, use_csls: bool,
              cnt_row: torch.Tensor, cnt_col: torch.Tensor, want_top3: bool = False):
    """Rank counters of sweep 2 (ops.eval_rank's band path): the sweep on the split operands with the fp32 deferral band,
    then the canonical re-score of the deferred elements on the fp32 rows; an overflowing band list is retried larger.
    There is no in-kernel chain fallback here (its verdicts come from tensor-core scores): past RANK_BAND_MAX_CAP
    deferred elements it raises."""
    Xr, Yr = _rows(X, "X"), _rows(Y, "Y")
    _need(cnt_row, torch.int32, "cnt_row", 1)
    _need(cnt_col, torch.int32, "cnt_col", 1)
    dev, st = Xr.device, current_stream()
    t3v = t3i = None
    if want_top3:
        _, nch = ops.sim_plan(n1, n2, X.split.shape[1])
        t3v = torch.empty((nch, n1, 4), dtype=torch.float32, device=dev)
        t3i = torch.empty((nch, n1, 4), dtype=torch.int32, device=dev)
    eps = rank_band_eps(xn, yn, Xr.shape[1])
    cap = max(ops.RANK_BAND_MIN_CAP, ops.RANK_BAND_PER_ROW * (n1 + n2))
    row_save, col_save = cnt_row.clone(), cnt_col.clone()
    while True:
        band = torch.empty((cap,), dtype=torch.int64, device=dev)
        band_cnt = torch.zeros((1,), dtype=torch.int32, device=dev)
        with ops._SweepTimer("sim_kernel<EpiRank>", n1, n2):
            call("snag_eval_rank_band", ptr(X.split), ptr(Y.split), ptr(xn), ptr(yn), ptr(nv1), ptr(nv2), ptr(g_row), ptr(g_col),
                 row_gid0, col_gid0, n1, n2, X.split.shape[1], int(use_csls), eps, ptr(cnt_row), ptr(cnt_col), ptr(t3v), ptr(t3i),
                 ptr(band), ptr(band_cnt), cap, st)
        call("snag_band_rescore_f32", ptr(Xr), ptr(Yr), Xr.shape[1], ptr(xn), ptr(yn), ptr(nv1), ptr(nv2), ptr(g_row),
             ptr(g_col), row_gid0, col_gid0, int(use_csls), ptr(band), ptr(band_cnt), cap, ptr(cnt_row), ptr(cnt_col), st)
        deferred = int(band_cnt.item()) & 0xFFFFFFFF
        LAST_RANK_INFO.clear()
        LAST_RANK_INFO.update(deferred=deferred, cap=cap, mode="band", eps=eps)
        if deferred <= cap:
            return t3v, t3i
        if cap >= RANK_BAND_MAX_CAP:
            raise SnagError(f"{deferred} elements of the fp32 rank sweep are within the error bound of a ground-truth "
                            f"distance (nearly all ties): more than the deferral list can hold")
        cnt_row.copy_(row_save)
        cnt_col.copy_(col_save)
        cap = min(RANK_BAND_MAX_CAP, max(cap * 8, round_up(deferred + deferred // 8, 1024)))


def rank_judge(X, Y, xn, yn, nv1, nv2, g_row, g_col, row_gid0: int, col_gid0: int, rk_stream, rk_stream_row, rk_cnt,
               R, Rp, C, Cp, row_ok, col_ok, eps: float, cnt_row: torch.Tensor, cnt_col: torch.Tensor):
    """ops.rank_judge with the deferred elements re-scored on the fp32 rows (snag_rank_judge + snag_band_rescore_f32)."""
    Xr, Yr = _rows(X, "X"), _rows(Y, "Y")
    _need(rk_stream, torch.int64, "rk_stream", 2)
    _need(rk_stream_row, torch.int32, "rk_stream_row", 2)
    _need(rk_cnt, torch.int32, "rk_cnt", 1)
    _need(row_ok, torch.uint8, "row_ok", 1)
    _need(col_ok, torch.uint8, "col_ok", 1)
    dev, st = Xr.device, current_stream()
    n_ctas, rk_cap = rk_stream.shape
    overflow = torch.zeros((1,), dtype=torch.int32, device=dev)
    cap = max(ops.RANK_BAND_MIN_CAP, ops.RANK_BAND_PER_ROW * (R.numel() + C.numel()))
    row_save, col_save = cnt_row.clone(), cnt_col.clone()
    while True:
        band = torch.empty((cap,), dtype=torch.int64, device=dev)
        band_cnt = torch.zeros((1,), dtype=torch.int32, device=dev)
        call("snag_rank_judge", ptr(rk_stream), ptr(rk_stream_row), ptr(rk_cnt), n_ctas, rk_cap, ptr(R), ptr(Rp), ptr(C), ptr(Cp),
             ptr(row_ok), ptr(col_ok), float(eps), row_gid0, col_gid0, ptr(cnt_row), ptr(cnt_col), ptr(band), ptr(band_cnt), cap,
             ptr(overflow), st)
        call("snag_band_rescore_f32", ptr(Xr), ptr(Yr), Xr.shape[1], ptr(xn), ptr(yn), ptr(nv1), ptr(nv2), ptr(g_row),
             ptr(g_col), row_gid0, col_gid0, 1, ptr(band), ptr(band_cnt), cap, ptr(cnt_row), ptr(cnt_col), st)
        deferred = int(band_cnt.item()) & 0xFFFFFFFF
        if deferred <= cap:
            return overflow, deferred
        cnt_row.copy_(row_save)
        cnt_col.copy_(col_save)
        cap = round_up(deferred + deferred // 8, 1024)


def rank_exhaustive(A, B, an, bn, nva, nvb, g, rows: torch.Tensor, a_gid0: int, b_gid0: int, use_csls: bool, swapped: bool,
                    cnt: torch.Tensor, n_b: int | None = None) -> None:
    """cnt[row] += canonical rank count of every listed row of A against the first n_b rows of B, on the fp32 rows."""
    Ar, Br = _rows(A, "A"), _rows(B, "B")
    _need(rows, torch.int32, "rows", 1)
    _need(cnt, torch.int32, "cnt", 1)
    if rows.numel() == 0:
        return
    call("snag_rank_exhaustive_f32", ptr(Ar), ptr(Br), Ar.shape[1], Br.shape[0] if n_b is None else n_b, ptr(an), ptr(bn),
         ptr(nva), ptr(nvb), ptr(g), ptr(rows), rows.numel(), a_gid0, b_gid0, int(use_csls), int(swapped), ptr(cnt),
         current_stream())


def rank_recount_rows(A, B, an, bn, nva, nvb, g_a, g_b, rows: torch.Tensor, a_gid0: int, b_gid0: int, n_b: int,
                      swapped: bool, eps: float) -> torch.Tensor:
    """ops.rank_recount_rows: the tensor-core sweep over the gathered sub-panel of split operands, the re-score of its
    deferred elements on the fp32 rows."""
    _rows(A, "A")
    Br = _rows(B, "B")
    _need(rows, torch.int32, "rows", 1)
    f = rows.numel()
    dev = Br.device
    cnt = torch.zeros((f,), dtype=torch.int32, device=dev)
    if f == 0:
        return cnt
    idx = rows.long()
    Af = A.index_select(0, idx)
    anf, nvaf, gf = an.index_select(0, idx), nva.index_select(0, idx), g_a.index_select(0, idx)
    gids = (rows + a_gid0).contiguous()
    scratch = torch.zeros((n_b,), dtype=torch.int32, device=dev)
    st = current_stream()
    cap = max(ops.RANK_BAND_MIN_CAP, ops.RANK_BAND_PER_ROW * (f + n_b))
    while True:
        band = torch.empty((cap,), dtype=torch.int64, device=dev)
        band_cnt = torch.zeros((1,), dtype=torch.int32, device=dev)
        with ops._SweepTimer("sim_kernel<EpiRank>[recount]", f, n_b):
            call("snag_eval_rank_band_rows", ptr(Af.split), ptr(B.split), ptr(anf), ptr(bn), ptr(nvaf), ptr(nvb), ptr(gf), ptr(g_b),
                 ptr(gids), b_gid0, f, n_b, Af.split.shape[1], 1, float(eps), ptr(cnt), ptr(scratch), ptr(band), ptr(band_cnt),
                 cap, st)
        call("snag_band_rescore_rows_f32", ptr(Af.rows), ptr(Br), Br.shape[1], ptr(anf), ptr(bn), ptr(nvaf), ptr(nvb), ptr(gf),
             ptr(g_b), ptr(gids), b_gid0, 1, int(swapped), ptr(band), ptr(band_cnt), cap, ptr(cnt), ptr(scratch), st)
        deferred = int(band_cnt.item()) & 0xFFFFFFFF
        if deferred <= cap:
            return cnt
        cnt.zero_()
        cap = round_up(deferred + deferred // 8, 1024)


def top3_rescore(X, Y, xn, yn, nv1, nv2, use_csls: bool, cand: torch.Tensor):
    """Canonical distances of each row's 4 merged nearest candidates on the fp32 rows, ascending (lower id first on ties):
    columns 0..2 are ret1..ret3 of the prediction file."""
    Xr, Yr = _rows(X, "X"), _rows(Y, "Y")
    _need(cand, torch.int32, "cand", 2)
    n_rows = cand.shape[0]
    oval = torch.empty((n_rows, 4), dtype=torch.float32, device=Xr.device)
    oidx = torch.empty((n_rows, 4), dtype=torch.int32, device=Xr.device)
    call("snag_top3_rescore_f32", ptr(Xr), ptr(Yr), Xr.shape[1], n_rows, ptr(xn), ptr(yn), ptr(nv1), ptr(nv2), int(use_csls),
         ptr(cand), ptr(oval), ptr(oidx), current_stream())
    return oval, oidx
