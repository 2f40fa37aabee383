"""Kernel backend of the fused --distance 1 evaluation (evaluate.evaluate_alignment_l1): the entry points
evaluate._align_ranks_steps calls, with cityblock semantics, over fp32 operands zero padded to Dp = round_up(D, 8)
(snag_b200/csrc/l1_sweep.cu). The xn / yn slots carry the rows' L1 norms, which scale the sweep's error bound.
There is no eval_rowcoltopk, so the generator takes its three-sweep path; sharding comes from the generator."""
from __future__ import annotations

import ctypes

import torch

from ._lib import KT, SnagError, call, current_stream, ptr
from .ops import _band_retry, _need, round_up
from .ops import num_sms, top4_merge, topk_merge_mean  # noqa: F401  (the generator calls them as be.*)

LAST_TOPK_INFO: dict = {}
LAST_RANK_INFO: dict = {}
BAND_MIN_CAP = 1 << 20
BAND_PER_ROW = 64            # initial deferral-list capacity per evaluated row + column
BAND_MAX_CAP = 1 << 28       # 2 GB of band entries: beyond that the input is nearly all ties
EXHAUSTIVE_BUDGET = 2.0e12   # fp64 element-ops the exhaustive neighbourhood completion may spend


def prep(emb: torch.Tensor, idx: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    """Rows emb[idx] as a zero-padded fp32 operand [n, round_up(D, 8)] (bit-identical values) and their L1 norms."""
    _need(emb, torch.float32, "emb", 2)
    n, d = idx.numel(), emb.shape[1]
    X = torch.zeros((n, round_up(d, 8)), dtype=torch.float32, device=emb.device)
    X[:, :d] = emb.index_select(0, idx)
    return X, X.abs().sum(1, dtype=torch.float64).to(torch.float32)


def _check(t: torch.Tensor, name: str) -> None:
    _need(t, torch.float32, name, 2)
    if t.shape[1] % 8:
        raise ValueError(f"{name}: width {t.shape[1]} is not a multiple of 8 (use l1.prep)")
    if t.data_ptr() % 16:
        raise ValueError(f"{name}: base pointer must be 16-byte aligned")


def n_lists(n1: int, n2: int, dp: int) -> int:
    nl = ctypes.c_int32()
    call("snag_l1_plan", n1, n2, dp, ctypes.byref(nl))
    return nl.value


def eval_rowtopk(X, Y, xn, yn, n1: int, n2: int, want_idx: bool = False):
    """Per-list candidate lists [n_lists, n1, KT] of c~ = 1 - d~ (ascending) and, with want_idx, their columns."""
    _check(X, "X")
    _check(Y, "Y")
    nl = n_lists(n1, n2, X.shape[1])
    part = torch.empty((nl, n1, KT), dtype=torch.float32, device=X.device)
    pidx = torch.empty((nl, n1, KT), dtype=torch.int32, device=X.device)
    call("snag_l1_rowtopk", ptr(X), ptr(Y), n1, n2, X.shape[1], ptr(part), ptr(pidx), current_stream())
    return (part, pidx) if want_idx else part


def topk_rescore(A, B, an, bn, cand_idx, cand_val, k: int, n_b: int, tag: str = "rows", outsider_bound=None):
    """Canonical CSLS neighbourhood means of the rows of A from their merged candidates; rows the candidates cannot vouch
    for are completed by an exhaustive canonical scan of the first n_b rows of B."""
    _check(A, "A")
    _check(B, "B")
    _need(cand_idx, torch.int32, "cand_idx", 2)
    _need(cand_val, torch.float32, "cand_val", 2)
    if outsider_bound is not None:
        raise ValueError("the L1 sweep lists see every column: no outsider bound")
    n_rows = cand_idx.shape[0]
    dev = A.device
    st = current_stream()
    nv = torch.empty((n_rows,), dtype=torch.float32, device=dev)
    flagged = torch.empty((n_rows,), dtype=torch.int32, device=dev)
    fcnt = torch.zeros((1,), dtype=torch.int32, device=dev)
    bmax = float(bn[:n_b].max().item())
    call("snag_l1_topk_rescore", ptr(A), ptr(B), A.shape[1], n_rows, ptr(an), bmax, ptr(cand_idx), ptr(cand_val), k, ptr(nv),
         ptr(flagged), ptr(fcnt), n_rows, st)
    n_flag = int(fcnt.item())
    info = {"flagged": n_flag, "unverified": 0}
    if n_flag:
        if float(n_flag) * n_b * A.shape[1] > EXHAUSTIVE_BUDGET:
            raise SnagError(f"{n_flag} {tag} L1 neighbourhoods could not be verified from {KT} candidates and their "
                            f"exhaustive completion exceeds the budget (plateaus of near-equal distances)")
        call("snag_l1_topk_exhaustive", ptr(A), ptr(B), A.shape[1], n_b, ptr(flagged), ptr(fcnt), n_rows, k, ptr(nv), st)
    LAST_TOPK_INFO[tag] = info
    return nv


def pair_score(X, Y, n: int, xn, yn, nv1, nv2, use_csls: bool):
    _check(X, "X")
    _check(Y, "Y")
    g = torch.empty((n,), dtype=torch.float32, device=X.device)
    call("snag_l1_pair_score", ptr(X), ptr(Y), X.shape[1], n, ptr(nv1), ptr(nv2), int(use_csls), ptr(g), current_stream())
    return g


def eval_rank(X, Y, xn, yn, nv1, nv2, g_row, g_col, row_gid0: int, col_gid0: int, n1: int, n2: int, use_csls: bool,
              cnt_row: torch.Tensor, cnt_col: torch.Tensor, want_top3: bool = False):
    """Rank counters accumulated into cnt_row / cnt_col: the sweep with its deferral band, then the canonical re-score of
    the deferred elements; a band list that overflows is retried with a larger one. Returns the per-list 4 nearest
    candidates ([n_lists, n1, 4] values -dist~, column gids) when want_top3, else (None, None)."""
    _check(X, "X")
    _check(Y, "Y")
    _need(cnt_row, torch.int32, "cnt_row", 1)
    _need(cnt_col, torch.int32, "cnt_col", 1)
    dev, st = X.device, current_stream()
    t3v = t3i = None
    if want_top3:
        nl = n_lists(n1, n2, X.shape[1])
        t3v = torch.empty((nl, n1, 4), dtype=torch.float32, device=dev)
        t3i = torch.empty((nl, n1, 4), dtype=torch.int32, device=dev)

    def attempt(band, band_cnt, cap):
        call("snag_l1_rank_band", ptr(X), ptr(Y), ptr(xn), ptr(yn), ptr(nv1), ptr(nv2), ptr(g_row), ptr(g_col), row_gid0,
             col_gid0, n1, n2, X.shape[1], int(use_csls), ptr(cnt_row), ptr(cnt_col), ptr(t3v), ptr(t3i), ptr(band),
             ptr(band_cnt), cap, st)
        call("snag_l1_band_rescore", ptr(X), ptr(Y), X.shape[1], ptr(nv1), ptr(nv2), ptr(g_row), ptr(g_col), row_gid0, col_gid0,
             int(use_csls), ptr(band), ptr(band_cnt), cap, ptr(cnt_row), ptr(cnt_col), st)

    deferred, cap = _band_retry(attempt, max(BAND_MIN_CAP, BAND_PER_ROW * (n1 + n2)), (cnt_row, cnt_col), grow=4,
                                max_cap=BAND_MAX_CAP, clamp=True)
    LAST_RANK_INFO.clear()
    LAST_RANK_INFO.update(deferred=deferred, cap=cap, mode="band")
    if deferred > cap:
        raise SnagError(f"{deferred} elements of the L1 rank sweep are within the error bound of a ground-truth "
                        f"distance (nearly all ties): more than the deferral list can hold")
    return t3v, t3i


def top3_rescore(X, Y, xn, yn, nv1, nv2, use_csls: bool, cand: torch.Tensor):
    """Canonical distances of each row's 4 merged nearest candidates (ids into Y), ascending with the lower id first on
    ties; rows whose candidates cannot vouch for the canonical top 3 are rescanned exhaustively. Columns 0..2 are
    ret1..ret3 of the prediction file."""
    _check(X, "X")
    _check(Y, "Y")
    _need(cand, torch.int32, "cand", 2)
    n_rows, n_b = cand.shape[0], yn.numel()
    dev = X.device
    oval = torch.empty((n_rows, 4), dtype=torch.float32, device=dev)
    oidx = torch.empty((n_rows, 4), dtype=torch.int32, device=dev)
    flagged = torch.empty((n_rows,), dtype=torch.int32, device=dev)
    fcnt = torch.zeros((1,), dtype=torch.int32, device=dev)
    ymax = float(yn.max().item())
    nvmax = float(nv2.abs().max().item()) if use_csls else 0.0
    call("snag_l1_top3_rescore", ptr(X), ptr(Y), X.shape[1], n_rows, n_b, ptr(xn), ymax, ptr(nv1), ptr(nv2), nvmax,
         int(use_csls), ptr(cand), ptr(oval), ptr(oidx), ptr(flagged), ptr(fcnt), current_stream())
    LAST_RANK_INFO["top3_rescanned"] = int(fcnt.item())
    return oval, oidx
