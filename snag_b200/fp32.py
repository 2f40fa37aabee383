"""Kernel backend of the fp32 evaluation (evaluate.evaluate_alignment(precision="fp32")) and of the fp32 link searches
(mining / seeds with precision="fp32"): the entry points evaluate._align_ranks_steps, mining.mutual_nearest and
seeds.topk_similarity_entries call, over the UNROUNDED fp32 rows.

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
from ._lib import call, current_stream, ptr
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


# ------------------------------------------------------------------------------------------------ forwards
# The entry points of snag_b200.ops with SplitOperand tables: the sweeps contract .split, the canonical re-scores read
# .rows (ops picks their snag_*_f32 kernels by the row dtype), and the tolerances come from the error model above.
def eval_rowtopk(X, Y, *args, **kw):
    return ops.eval_rowtopk(X.split, Y.split, *args, **kw)


def eval_rowcoltopk(X, Y, *args, **kw):
    return ops.eval_rowcoltopk(X.split, Y.split, *args, **kw)


def eval_onepass(X, Y, *args, **kw):
    return ops.eval_onepass(X.split, Y.split, *args, **kw)


def topk_rescore(A, B, an, bn, cand_idx, cand_val, k: int, n_b: int, tag: str = "rows", want_best: bool = False,
                 outsider_bound=None):
    return ops.topk_rescore(A.rows, B.rows, an, bn, cand_idx, cand_val, k, n_b, tag, want_best=want_best,
                            outsider_bound=outsider_bound, margin=_error_scale(an, bn, A.shape[1]), info=LAST_TOPK_INFO)


def pair_score(X, Y, *args, **kw):
    return ops.pair_score(X.rows, Y.rows, *args, **kw)


def pairs_dot(X, Y, *args):
    return ops.pairs_dot(X.rows, Y.rows, *args)


def eval_rank(X, Y, xn, yn, *args, **kw):
    return ops.eval_rank(X.split, Y.split, xn, yn, *args, **kw, eps=rank_band_eps(xn, yn, X.shape[1]),
                         canon=(X.rows, Y.rows), info=LAST_RANK_INFO)


def rank_judge(X, Y, *args, **kw):
    return ops.rank_judge(X.rows, Y.rows, *args, **kw)


def rank_exhaustive(A, B, *args, **kw):
    return ops.rank_exhaustive(A.rows, B.rows, *args, **kw)


def rank_recount_rows(A, B, *args, **kw):
    return ops.rank_recount_rows(A.split, B.split, *args, **kw, canon=(A.rows, B.rows))


def top3_rescore(X, Y, *args, **kw):
    return ops.top3_rescore(X.rows, Y.rows, *args, **kw)
