"""Thin torch-tensor wrappers over the C ABI: shape/dtype/contiguity validation in Python, pointers and
the current CUDA stream passed down, return codes turned into exceptions. No compute happens here."""
from __future__ import annotations

import torch

from . import _lib
from ._lib import KT, SnagError, call, current_stream, ptr


def _need(t: torch.Tensor, dtype, name: str, ndim: int | None = None) -> None:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise SnagError(f"{name} must live on a CUDA device: snag_b200 has no CPU path")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if ndim is not None and t.dim() != ndim:
        raise ValueError(f"{name} must be {ndim}-D, got shape {tuple(t.shape)}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")


def round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def num_sms() -> int:
    """SMs of the current device = persistent CTAs of a fused sweep (148 on a B200)."""
    return int(_lib.load().snag_num_sms())


def sim_plan(n_rows: int, n_cols: int, dpad: int) -> tuple[int, int]:
    """(tiles_per_chunk, n_lists) of an [n_rows x n_cols] sweep; n_lists partial lists per row are written."""
    return _lib.sim_plan(n_rows, n_cols, dpad)


# ------------------------------------------------------------------------------------------------ prologue
def prep_bf16(emb: torch.Tensor, idx: torch.Tensor | None = None, normalize: bool = True,
              rows_pad_to: int = 1, out: torch.Tensor | None = None) -> tuple[torch.Tensor, torch.Tensor]:
    """(gather ->) L2-normalise -> bf16, zero padded to a multiple of 64 columns; plus ||row||^2 (fp32) of the
    rounded rows. Returns (operand [n_pad, Dpad] bf16, norm2 [n] fp32); rows n..n_pad are zero.
    `out` (bf16 [>=n, Dpad], contiguous) receives the rows instead of a fresh allocation; its remaining rows are
    left untouched."""
    _need(emb, torch.float32, "emb", 2)
    n = emb.shape[0] if idx is None else idx.numel()
    if idx is not None:
        _need(idx, torch.int64, "idx", 1)
    if n == 0:
        raise ValueError("empty operand")
    d = emb.shape[1]
    dpad = round_up(d, 64)
    n_pad = round_up(n, rows_pad_to)
    if out is not None:
        _check_operand(out, "out")
        if out.shape[0] < n or out.shape[1] != dpad:
            raise ValueError(f"out must be [>= {n}, {dpad}], got {tuple(out.shape)}")
    elif n_pad == n:
        out = torch.empty((n_pad, dpad), dtype=torch.bfloat16, device=emb.device)
    else:
        out = torch.zeros((n_pad, dpad), dtype=torch.bfloat16, device=emb.device)
    norm2 = torch.empty((n,), dtype=torch.float32, device=emb.device)
    call("snag_prep_bf16", ptr(emb), emb.stride(0), ptr(idx), n, d, int(normalize), ptr(out), dpad, ptr(norm2),
         current_stream())
    return out, norm2


def _ptr_array(tensors):
    import ctypes
    arr = (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
    return arr


def joint_fuse_fwd(embs, w_ent: torch.Tensor | None, w_glob: torch.Tensor | None, want_joint: bool = True,
                   want_fz: bool = True):
    """(joint, joint_fz) [N, sum d_m] of model/SNAG_tools.py:44-49 from the M modality tables (fp32 [N, d_m])."""
    import ctypes
    if not 1 <= len(embs) <= 6:
        raise ValueError("1..6 modality tables")
    for t in embs:
        _need(t, torch.float32, "emb", 2)
    N = embs[0].shape[0]
    if any(t.shape[0] != N for t in embs):
        raise ValueError("modality tables must have the same number of rows")
    M = len(embs)
    widths = (ctypes.c_int32 * M)(*[int(t.shape[1]) for t in embs])
    tot = sum(int(t.shape[1]) for t in embs)
    if want_joint:
        _need(w_ent, torch.float32, "w_ent", 2)
        if w_ent.shape[0] != N or w_ent.shape[1] < M:
            raise ValueError("w_ent must be [N, >= M]")
    if want_fz:
        _need(w_glob, torch.float32, "w_glob", 1)
        if w_glob.numel() < M:
            raise ValueError("w_glob must have >= M entries")
    joint = torch.empty((N, tot), dtype=torch.float32, device=embs[0].device) if want_joint else None
    fz = torch.empty((N, tot), dtype=torch.float32, device=embs[0].device) if want_fz else None
    call("snag_joint_fuse_fwd", _ptr_array(embs), widths, M, N, ptr(w_ent) if want_joint else None,
         w_ent.stride(0) if want_joint else 0, ptr(w_glob) if want_fz else None, ptr(joint), ptr(fz), tot, current_stream())
    return joint, fz


def joint_fuse_bwd(embs, w_ent, w_glob, d_joint, d_fz):
    """Gradients of joint_fuse_fwd: (list of d_emb [N, d_m], d_w_ent [N, w_ent.shape[1]] or None, d_w_glob [len] or None)."""
    import ctypes
    M, N = len(embs), embs[0].shape[0]
    widths = (ctypes.c_int32 * M)(*[int(t.shape[1]) for t in embs])
    tot = sum(int(t.shape[1]) for t in embs)
    for g, nm in ((d_joint, "d_joint"), (d_fz, "d_joint_fz")):
        if g is not None:
            _need(g, torch.float32, nm, 2)
            if tuple(g.shape) != (N, tot):
                raise ValueError(f"{nm} must be [N, sum of widths]")
    d_embs = [torch.empty_like(t) for t in embs]
    d_w_ent = torch.zeros_like(w_ent) if d_joint is not None else None
    d_w_glob = torch.zeros_like(w_glob) if d_fz is not None else None
    call("snag_joint_fuse_bwd", _ptr_array(embs), _ptr_array(d_embs), widths, M, N,
         ptr(w_ent) if d_joint is not None else None, w_ent.stride(0) if d_joint is not None else 0,
         ptr(w_glob) if d_fz is not None else None, ptr(d_joint), ptr(d_fz), tot, ptr(d_w_ent), ptr(d_w_glob), current_stream())
    return d_embs, d_w_ent, d_w_glob


def normalize_bwd_scatter(emb: torch.Tensor, idx: torch.Tensor | None, dz: torch.Tensor, demb: torch.Tensor,
                          normalize: bool = True) -> None:
    """demb[idx[r]] += d/d emb[idx[r]] of F.normalize(emb[idx[r]]) . dz[r] — the backward of prep_bf16's gather +
    normalise, accumulated in place (demb fp32 [N, D], same layout as emb). dz is [>= n, >= D] or, as the partial sums
    of the fused backward's column splits, [n_parts, >= n, >= D] (added in split order)."""
    _need(emb, torch.float32, "emb", 2)
    _need(demb, torch.float32, "demb", 2)
    if not isinstance(dz, torch.Tensor) or dz.dtype != torch.float32 or not dz.is_cuda or dz.dim() not in (2, 3) or dz.stride(-1) != 1:
        raise TypeError("dz must be a CUDA fp32 tensor [n, D] or [n_parts, n, D] with contiguous rows")
    if idx is not None:
        _need(idx, torch.int64, "idx", 1)
    n = emb.shape[0] if idx is None else idx.numel()
    n_parts, part_stride = (1, 0) if dz.dim() == 2 else (dz.shape[0], dz.stride(0))
    if dz.shape[-2] < n or dz.shape[-1] < emb.shape[1] or demb.shape != emb.shape:
        raise ValueError("normalize_bwd_scatter: shape mismatch")
    call("snag_normalize_bwd_scatter", ptr(emb), emb.stride(0), ptr(idx), n, emb.shape[1], int(normalize), ptr(dz),
         dz.stride(-2), n_parts, part_stride, ptr(demb), demb.stride(0), current_stream())


def _check_operand(t: torch.Tensor, name: str) -> None:
    _need(t, torch.bfloat16, name, 2)
    if t.shape[1] % 64:
        raise ValueError(f"{name}: width {t.shape[1]} is not a multiple of 64 (use prep_bf16)")
    if t.data_ptr() % 128:
        raise ValueError(f"{name}: base pointer must be 128-byte aligned")


def _suffix(X: torch.Tensor, Y: torch.Tensor, names: str = "XY") -> str:
    """Suffix of the canonical entry points for the row type of X and Y: "" (snag_X) for bf16 operands (prep_bf16),
    "_f32" (snag_X_f32) for the fp32 rows of fp32.prep ([n, multiple of 64], 16-byte aligned)."""
    for t, nm in ((X, names[0]), (Y, names[1])):
        if isinstance(t, torch.Tensor) and t.dtype == torch.float32:
            _need(t, torch.float32, nm, 2)
            if t.shape[1] % 64 or t.data_ptr() % 16:
                raise ValueError(f"{nm}: fp32 rows must be [n, multiple of 64] and 16-byte aligned")
        else:
            _check_operand(t, nm)
    if X.dtype != Y.dtype:
        raise TypeError(f"{names[0]} and {names[1]} must have the same dtype")
    return "" if X.dtype == torch.bfloat16 else "_f32"


def _band_retry(attempt, cap: int, counters: tuple, grow: int = 1, max_cap: int | None = None, clamp: bool = False,
                sync: bool = True):
    """The deferral-list protocol of the band sweeps. attempt(band, band_cnt, cap) enqueues a sweep or judge that lists
    the elements it cannot decide in `band` (band_cnt counts them all, also those past cap) and their canonical
    re-score, both adding to `counters`. After an overflow the counters are restored and the attempt repeats with
    max(grow x cap, 9/8 of the count rounded up to 1024) entries, clamped to max_cap when `clamp`. Returns (deferred,
    cap) of the last attempt; deferred > cap (counters restored) when the list would have to grow past max_cap or,
    clamped, a list of max_cap overflowed. sync=False: one attempt, no host synchronisation (CUDA-graph capture);
    returns the DEVICE band_cnt and cap, and the caller must check deferred <= cap before trusting the counters."""
    dev = counters[0].device
    saved = [t.clone() for t in counters] if sync else None
    while True:
        band = torch.empty((cap,), dtype=torch.int64, device=dev)
        band_cnt = torch.zeros((1,), dtype=torch.int32, device=dev)
        attempt(band, band_cnt, cap)
        if not sync:
            return band_cnt, cap
        deferred = int(band_cnt.item()) & 0xFFFFFFFF
        if deferred <= cap:
            return deferred, cap
        for t, s in zip(counters, saved):
            t.copy_(s)
        grown = max(grow * cap, round_up(deferred + deferred // 8, 1024))
        if max_cap is not None and (cap >= max_cap if clamp else grown > max_cap):
            return deferred, cap
        cap = min(grown, max_cap) if clamp else grown


# ------------------------------------------------------------------------------------------------ eval sweeps
def sim_write(X: torch.Tensor, Y: torch.Tensor, xn: torch.Tensor | None, yn: torch.Tensor | None, n1: int, n2: int,
              mode: int) -> torch.Tensor:
    _check_operand(X, "X")
    _check_operand(Y, "Y")
    if mode == 1:
        _need(xn, torch.float32, "xn", 1)
        _need(yn, torch.float32, "yn", 1)
    out = torch.empty((n1, n2), dtype=torch.float32, device=X.device)
    with _SweepTimer("sim_kernel<EpiWrite>", n1, n2, X.shape[1]):
        call("snag_sim_write", ptr(X), ptr(Y), ptr(xn), ptr(yn), n1, n2, X.shape[1], mode, ptr(out), out.stride(0),
             current_stream())
    return out


def sim_mainloop_only(X: torch.Tensor, Y: torch.Tensor, n1: int, n2: int) -> None:
    """Measurement aid: the sweep without any epilogue (see snag_sim_mainloop_only)."""
    _check_operand(X, "X")
    _check_operand(Y, "Y")
    call("snag_sim_mainloop_only", ptr(X), ptr(Y), n1, n2, X.shape[1], current_stream())


# Measurement hook: when bench.py sets this to a list, every fused-sweep launch is bracketed by CUDA events on the
# launching stream and (name, start, end, rows, cols, depth) is appended (depth = contraction width, None = the
# caller knows it). None (the default) adds no events.
SWEEP_EVENT_SINK = None


class _SweepTimer:
    def __init__(self, name: str, rows: int, cols: int, depth: int | None = None):
        self.args = (name, rows, cols, depth) if SWEEP_EVENT_SINK is not None else None

    def __enter__(self):
        if self.args is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if self.args is not None and exc[0] is None:
            self.e1.record()
            SWEEP_EVENT_SINK.append((self.args[0], self.e0, self.e1, self.args[1], self.args[2], self.args[3]))


def eval_rowtopk(X, Y, xn, yn, n1: int, n2: int, want_idx: bool = False):
    """Per-list candidate lists [n_lists, n1, KT] of c = 1 - d for every row of X against the rows of Y; with
    want_idx also the column of every candidate (int32, -1 = padding): returns part or (part, part_idx)."""
    _check_operand(X, "X")
    _check_operand(Y, "Y")
    _need(xn, torch.float32, "xn", 1)
    _need(yn, torch.float32, "yn", 1)
    _, nch = sim_plan(n1, n2, X.shape[1])
    part = torch.empty((nch, n1, KT), dtype=torch.float32, device=X.device)
    pidx = torch.empty((nch, n1, KT), dtype=torch.int32, device=X.device) if want_idx else None
    with _SweepTimer("sim_kernel<EpiRowTopK>", n1, n2):
        call("snag_eval_rowtopk", ptr(X), ptr(Y), ptr(xn), ptr(yn), n1, n2, X.shape[1], ptr(part), ptr(pidx),
             current_stream())
    return (part, pidx) if want_idx else part


def col_threshold(cand: torch.Tensor, k: int, yn: torch.Tensor):
    """(colthr, colb) of the two-sweep evaluation from the merged sample lists [n, KT] (see snag_col_threshold)."""
    _need(cand, torch.float32, "cand", 2)
    _need(yn, torch.float32, "yn", 1)
    n = cand.shape[0]
    colthr = torch.empty((n,), dtype=torch.float32, device=cand.device)
    colb = torch.empty((n,), dtype=torch.float32, device=cand.device)
    call("snag_col_threshold", ptr(cand), n, k, ptr(yn), ptr(colthr), ptr(colb), current_stream())
    return colthr, colb


HALF_PREFILTER_NORM2_MAX = 1.05    # SNAG_HALF_PREFILTER_NORM2_MAX of the library


def eval_rowcoltopk(X, Y, xn, yn, n1: int, n2: int, colthr, colb, cta_cap: int, rowthr: torch.Tensor | None = None,
                    norm2_max: float | None = None):
    """One sweep for both CSLS directions: returns (row candidate lists [n_lists, n1, KT], their columns (int32, same
    shape), per-CTA candidate streams int64 [n_ctas, cta_cap] (low word column, high word c bits), the row of every
    stream entry int32 [n_ctas, cta_cap], stream_cnt int32 [n_ctas])."""
    _check_operand(X, "X")
    _check_operand(Y, "Y")
    _need(xn, torch.float32, "xn", 1)
    _need(yn, torch.float32, "yn", 1)
    _need(colthr, torch.float32, "colthr", 1)
    _need(colb, torch.float32, "colb", 1)
    if rowthr is not None:
        _need(rowthr, torch.float32, "rowthr", 1)
        if rowthr.numel() < n1:
            raise ValueError("rowthr needs one entry per row")
    _, nch = sim_plan(n1, n2, X.shape[1])
    n_ctas = num_sms()
    part = torch.empty((nch, n1, KT), dtype=torch.float32, device=X.device)
    pidx = torch.empty((nch, n1, KT), dtype=torch.int32, device=X.device)
    stream = torch.empty((n_ctas, cta_cap), dtype=torch.int64, device=X.device)
    stream_row = torch.empty((n_ctas, cta_cap), dtype=torch.int32, device=X.device)
    stream_cnt = torch.zeros((n_ctas,), dtype=torch.int32, device=X.device)
    with _SweepTimer("sim_kernel<EpiRowColTopK>", n1, n2):
        if norm2_max is None:
            norm2_max = float(torch.maximum(xn.max(), yn.max()).item())
        call("snag_eval_rowcoltopk", ptr(X), ptr(Y), ptr(xn), ptr(yn), n1, n2, X.shape[1], ptr(part), ptr(pidx), ptr(rowthr),
             ptr(colthr), ptr(colb), ptr(stream), ptr(stream_row), ptr(stream_cnt), cta_cap, float(norm2_max), current_stream())
    return part, pidx, stream, stream_row, stream_cnt


def spec_bounds(cand: torch.Tensor, cdiag: torch.Tensor, k: int, shift: float, delta: float):
    """(lo, hi) of every entity's CSLS neighbourhood mean from its merged sample list [n, KT] and the canonical c of
    its own pair (see snag_spec_bounds): lo is a guaranteed lower bound, hi an extrapolated guess."""
    _need(cand, torch.float32, "cand", 2)
    _need(cdiag, torch.float32, "cdiag", 1)
    n = cand.shape[0]
    if cand.shape[1] != KT or cdiag.numel() != n:
        raise ValueError("cand must be [n, SNAG_KT] and cdiag [n]")
    lo = torch.empty((n,), dtype=torch.float32, device=cand.device)
    hi = torch.empty((n,), dtype=torch.float32, device=cand.device)
    call("snag_spec_bounds", ptr(cand), n, k, ptr(cdiag), float(shift), float(delta), ptr(lo), ptr(hi), current_stream())
    return lo, hi


def eval_onepass(X, Y, xn, yn, n1: int, n2: int, colthr, colb, cta_cap: int, rowthr, rk_r, rk_rp, rk_c, rk_cp, rk_cap: int,
                 norm2_max: float | None = None):
    """eval_rowcoltopk that also streams the rank candidates (snag_eval_onepass). Returns the five outputs of
    eval_rowcoltopk followed by (rk_stream int64 [n_ctas, rk_cap], rk_stream_row int32 [n_ctas, rk_cap], rk_cnt int32 [n_ctas])."""
    _check_operand(X, "X")
    _check_operand(Y, "Y")
    for name, t, cnt in (("xn", xn, n1), ("yn", yn, n2), ("colthr", colthr, n2), ("colb", colb, n2), ("rowthr", rowthr, n1),
                         ("rk_r", rk_r, n1), ("rk_rp", rk_rp, n1), ("rk_c", rk_c, n2), ("rk_cp", rk_cp, n2)):
        _need(t, torch.float32, name, 1)
        if t.numel() < cnt:
            raise ValueError(f"{name} needs {cnt} entries")
    _, nch = sim_plan(n1, n2, X.shape[1])
    n_ctas = num_sms()
    dev = X.device
    part = torch.empty((nch, n1, KT), dtype=torch.float32, device=dev)
    pidx = torch.empty((nch, n1, KT), dtype=torch.int32, device=dev)
    stream = torch.empty((n_ctas, cta_cap), dtype=torch.int64, device=dev)
    stream_row = torch.empty((n_ctas, cta_cap), dtype=torch.int32, device=dev)
    stream_cnt = torch.zeros((n_ctas,), dtype=torch.int32, device=dev)
    rk_stream = torch.empty((n_ctas, rk_cap), dtype=torch.int64, device=dev)
    rk_stream_row = torch.empty((n_ctas, rk_cap), dtype=torch.int32, device=dev)
    rk_cnt = torch.zeros((n_ctas,), dtype=torch.int32, device=dev)
    if norm2_max is None:
        norm2_max = float(torch.maximum(xn.max(), yn.max()).item())
    with _SweepTimer("sim_kernel<EpiOnePass>", n1, n2):
        call("snag_eval_onepass", ptr(X), ptr(Y), ptr(xn), ptr(yn), n1, n2, X.shape[1], ptr(part), ptr(pidx), ptr(rowthr),
             ptr(colthr), ptr(colb), ptr(stream), ptr(stream_row), ptr(stream_cnt), cta_cap, ptr(rk_r), ptr(rk_rp), ptr(rk_c),
             ptr(rk_cp), ptr(rk_stream), ptr(rk_stream_row), ptr(rk_cnt), rk_cap, float(norm2_max), current_stream())
    return part, pidx, stream, stream_row, stream_cnt, rk_stream, rk_stream_row, rk_cnt


def rank_judge(X, Y, xn, yn, nv1, nv2, g_row, g_col, row_gid0: int, col_gid0: int, rk_stream, rk_stream_row, rk_cnt,
               R, Rp, C, Cp, row_ok, col_ok, eps: float, cnt_row: torch.Tensor, cnt_col: torch.Tensor):
    """Settle the streamed rank candidates of eval_onepass against the final constants (snag_rank_judge) and re-score
    the elements inside the band canonically (snag_band_rescore); counts are accumulated into cnt_row / cnt_col.
    X, Y are the canonical rows of the re-score (bf16 operands or fp32 rows).
    Returns (overflow int32[1] device tensor — a rank stream was full, the counts are incomplete —, deferred count)."""
    sfx = _suffix(X, Y)
    _need(rk_stream, torch.int64, "rk_stream", 2)
    _need(rk_stream_row, torch.int32, "rk_stream_row", 2)
    _need(rk_cnt, torch.int32, "rk_cnt", 1)
    for name, t in (("R", R), ("Rp", Rp), ("C", C), ("Cp", Cp)):
        _need(t, torch.float32, name, 1)
    _need(row_ok, torch.uint8, "row_ok", 1)
    _need(col_ok, torch.uint8, "col_ok", 1)
    n_ctas, rk_cap = rk_stream.shape
    st = current_stream()
    overflow = torch.zeros((1,), dtype=torch.int32, device=X.device)

    def attempt(band, band_cnt, cap):
        call("snag_rank_judge", ptr(rk_stream), ptr(rk_stream_row), ptr(rk_cnt), n_ctas, rk_cap, ptr(R), ptr(Rp), ptr(C), ptr(Cp),
             ptr(row_ok), ptr(col_ok), float(eps), row_gid0, col_gid0, ptr(cnt_row), ptr(cnt_col), ptr(band), ptr(band_cnt), cap,
             ptr(overflow), st)
        call("snag_band_rescore" + sfx, ptr(X), ptr(Y), X.shape[1], ptr(xn), ptr(yn), ptr(nv1), ptr(nv2), ptr(g_row),
             ptr(g_col), row_gid0, col_gid0, 1, ptr(band), ptr(band_cnt), cap, ptr(cnt_row), ptr(cnt_col), st)

    deferred, _ = _band_retry(attempt, max(RANK_BAND_MIN_CAP, RANK_BAND_PER_ROW * (R.numel() + C.numel())), (cnt_row, cnt_col))
    return overflow, deferred


def rank_exhaustive(A, B, an, bn, nva, nvb, g, rows: torch.Tensor, a_gid0: int, b_gid0: int, use_csls: bool, swapped: bool,
                    cnt: torch.Tensor, n_b: int | None = None) -> None:
    """cnt[row] += canonical rank count of every listed row of A against the first n_b rows of B (snag_rank_exhaustive)."""
    sfx = _suffix(A, B, "AB")
    _need(rows, torch.int32, "rows", 1)
    _need(cnt, torch.int32, "cnt", 1)
    if rows.numel() == 0:
        return
    call("snag_rank_exhaustive" + sfx, ptr(A), ptr(B), A.shape[1], B.shape[0] if n_b is None else n_b, ptr(an), ptr(bn),
         ptr(nva), ptr(nvb), ptr(g), ptr(rows), rows.numel(), a_gid0, b_gid0, int(use_csls), int(swapped), ptr(cnt), current_stream())


def rank_recount_rows(A, B, an, bn, nva, nvb, g_a, g_b, rows: torch.Tensor, a_gid0: int, b_gid0: int, n_b: int,
                      swapped: bool, eps: float, canon: tuple | None = None) -> torch.Tensor:
    """Rank counts of the listed rows of A against the first n_b rows of B by a tensor-core sweep over the gathered
    sub-panel (snag_eval_rank_band_rows + snag_band_rescore_rows): the recount of entities whose one-pass guess failed.
    A = sources and B = targets (swapped False: l2r ranks of the listed sources), or A = targets and B = sources
    (swapped True: r2l ranks of the listed targets). an / nva / g_a are indexed like A, bn / nvb / g_b like B.
    canon: the canonical rows (of A, of B) of the re-score when they are not A and B (the fp32 rows of split operands).
    Returns int32 [len(rows)]."""
    _check_operand(A, "A")
    _check_operand(B, "B")
    Ac, Bc = (A, B) if canon is None else canon
    sfx = _suffix(Ac, Bc, "AB")
    _need(rows, torch.int32, "rows", 1)
    f = rows.numel()
    dev = A.device
    cnt = torch.zeros((f,), dtype=torch.int32, device=dev)
    if f == 0:
        return cnt
    idx = rows.long()
    Af = A.index_select(0, idx)
    Acf = Af if canon is None else Ac.index_select(0, idx)
    anf, nvaf, gf = an.index_select(0, idx), nva.index_select(0, idx), g_a.index_select(0, idx)
    gids = (rows + a_gid0).contiguous()
    scratch = torch.zeros((n_b,), dtype=torch.int32, device=dev)
    st = current_stream()

    def attempt(band, band_cnt, cap):
        with _SweepTimer("sim_kernel<EpiRank>[recount]", f, n_b):
            call("snag_eval_rank_band_rows", ptr(Af), ptr(B), ptr(anf), ptr(bn), ptr(nvaf), ptr(nvb), ptr(gf), ptr(g_b), ptr(gids),
                 b_gid0, f, n_b, A.shape[1], 1, float(eps), ptr(cnt), ptr(scratch), ptr(band), ptr(band_cnt), cap, st)
        call("snag_band_rescore_rows" + sfx, ptr(Acf), ptr(Bc), Bc.shape[1], ptr(anf), ptr(bn), ptr(nvaf), ptr(nvb), ptr(gf), ptr(g_b),
             ptr(gids), b_gid0, 1, int(swapped), ptr(band), ptr(band_cnt), cap, ptr(cnt), ptr(scratch), st)

    _band_retry(attempt, max(RANK_BAND_MIN_CAP, RANK_BAND_PER_ROW * (f + n_b)), (cnt,))
    return cnt


def col_cand_reduce(stream: torch.Tensor, stream_row: torch.Tensor, stream_cnt: torch.Tensor, n_cols: int, k: int):
    """Bucket the per-CTA candidate streams by column and keep each column's KT best candidates.
    Returns (cand_val [n_cols, KT] ascending, cand_idx [n_cols, KT] rows, overflow int32[1] device tensor)."""
    _need(stream, torch.int64, "stream", 2)
    _need(stream_row, torch.int32, "stream_row", 2)
    _need(stream_cnt, torch.int32, "stream_cnt", 1)
    dev = stream.device
    n_ctas, cta_cap = stream.shape
    st = current_stream()
    hist = torch.zeros((n_cols,), dtype=torch.int32, device=dev)
    overflow = torch.zeros((1,), dtype=torch.int32, device=dev)
    call("snag_col_cand_hist", ptr(stream), ptr(stream_cnt), n_ctas, cta_cap, ptr(hist), ptr(overflow), st)
    incl = torch.cumsum(hist, 0, dtype=torch.int64)
    offs = (incl - hist).contiguous()
    total = int(min(int(stream_cnt.clamp(max=cta_cap).sum().item()), n_ctas * cta_cap))
    vals = torch.empty((max(total, 1),), dtype=torch.float32, device=dev)
    rows = torch.empty((max(total, 1),), dtype=torch.int32, device=dev)
    cursor = torch.zeros((n_cols,), dtype=torch.int32, device=dev)
    call("snag_col_cand_scatter", ptr(stream), ptr(stream_row), ptr(stream_cnt), n_ctas, cta_cap, ptr(offs), ptr(cursor),
         ptr(vals), ptr(rows), st)
    cand_val = torch.empty((n_cols, KT), dtype=torch.float32, device=dev)
    cand_idx = torch.empty((n_cols, KT), dtype=torch.int32, device=dev)
    call("snag_col_cand_finalize", ptr(offs), ptr(hist), ptr(vals), ptr(rows), n_cols, k, None, ptr(cand_val), ptr(cand_idx),
         ptr(overflow), st)
    return cand_val, cand_idx, overflow


def mutual_nn(X, Y, xn, yn, n1: int, n2: int, colb: torch.Tensor):
    """Fused argmin sweep (snag_mutual_nn): returns (row_val [L, n1], row_idx [L, n1], colkey int64 [n2])."""
    _check_operand(X, "X")
    _check_operand(Y, "Y")
    _need(xn, torch.float32, "xn", 1)
    _need(yn, torch.float32, "yn", 1)
    _need(colb, torch.float32, "colb", 1)
    _, nl = sim_plan(n1, n2, X.shape[1])
    row_val = torch.empty((nl, n1), dtype=torch.float32, device=X.device)
    row_idx = torch.empty((nl, n1), dtype=torch.int32, device=X.device)
    colkey = torch.full((n2,), -1, dtype=torch.int64, device=X.device)          # all ones
    with _SweepTimer("sim_kernel<EpiMutualNN>", n1, n2, X.shape[1]):
        call("snag_mutual_nn", ptr(X), ptr(Y), ptr(xn), ptr(yn), n1, n2, X.shape[1], ptr(colb), ptr(colkey), ptr(row_val),
             ptr(row_idx), current_stream())
    return row_val, row_idx, colkey


def topk_merge_mean(part: torch.Tensor, k: int, want_nv: bool = True, want_cand: bool = False,
                    part_idx: torch.Tensor | None = None):
    """Merge per-list candidate lists. Returns (nv, cand) — or (nv, cand, cand_idx) when the lists' ids are passed."""
    _need(part, torch.float32, "part", 3)
    if part.shape[2] != KT:
        raise ValueError("candidate lists must have SNAG_KT entries")
    if not 1 <= k <= KT:
        raise SnagError(f"csls_k={k} unsupported: the fused CSLS path keeps {KT} candidates per row")
    if part_idx is not None:
        _need(part_idx, torch.int32, "part_idx", 3)
        want_cand = True
    n_lists, n_rows = part.shape[0], part.shape[1]
    nv = torch.empty((n_rows,), dtype=torch.float32, device=part.device) if want_nv else None
    cand = torch.empty((n_rows, KT), dtype=torch.float32, device=part.device) if want_cand else None
    cidx = torch.empty((n_rows, KT), dtype=torch.int32, device=part.device) if part_idx is not None else None
    call("snag_topk_merge_mean", ptr(part), ptr(part_idx), n_lists, n_rows, k, ptr(nv), ptr(cand), ptr(cidx),
         current_stream())
    return (nv, cand) if part_idx is None else (nv, cand, cidx)


# Worst |s_tensor_core - s_canonical| (canonical = fp64 index-order dot rounded once) measured over 2 x 1.07e9 pairs of
# unit rows built to provoke it (tests/test_eval_baseline_gpu.py::test_band_epsilon_covers_tensor_core_error_on_1e9_pairs:
# exact duplicates of all-positive and constant rows, where every partial sum is as large as it can be):
#   1.03e-5 at Dpad = 1216, 1.38e-5 at Dpad = 1856
# i.e. it grows about linearly with the number of accumulation steps (the tensor core's fp32 accumulation truncates):
# 8.4e-9 and 7.4e-9 per contraction element, bounded here by 9e-9; on typical (mixed-sign, s << 1) pairs it stays below
# 1e-6. Every tolerance that separates "the tensor cores decided" from "re-score canonically" is 4 x that bound plus the
# fp32 chain's roundings.
TC_DOT_ERR_PER_K = 9e-9
TC_MARGIN_FLOOR = 4e-6


def tc_margin(dpad: int, norm: float = 1.0) -> float:
    """Half-width (in units of the dot product s) inside which a tensor-core verdict is not trusted, for operands of
    width `dpad` whose rows have at most `norm` = ||x|| ||y||: 4 x the measured worst accumulation error + 1e-6 for the
    roundings of the reference's fp32 chain and of the per-row / per-column thresholds."""
    return max(TC_MARGIN_FLOOR, 4.0 * TC_DOT_ERR_PER_K * dpad * max(1.0, norm) + 1e-6)


# |c_tensor_core - c_canonical| = 2 |s_tc - s_canonical| + two fp32 roundings: the neighbourhood verification works in c
TOPK_VERIFY_DELTA = 2.0
TOPK_EXHAUSTIVE_BUDGET = 4.0e12     # bf16 multiply-adds the exhaustive completion may spend (~1 s of fp64 work on a B200)
LAST_TOPK_INFO: dict = {}


def topk_rescore(A, B, an, bn, cand_idx: torch.Tensor, cand_val: torch.Tensor, k: int, n_b: int, tag: str = "rows",
                 want_best: bool = False, outsider_bound: torch.Tensor | None = None, norm_bound: float | None = None,
                 lazy: bool = False, margin: float | None = None, info: dict | None = None):
    """Canonical CSLS neighbourhood means of the rows of A from their KT tensor-core candidates (rows of B; bf16
    operands or fp32 rows); rows the candidates cannot vouch for are completed by an exhaustive scan of B (within
    TOPK_EXHAUSTIVE_BUDGET; beyond it the candidate-based value stays and the count is reported in
    info[tag]['unverified'], info defaulting to LAST_TOPK_INFO).
    margin: the verification half-width in s of the caller's error model (default: tc_margin of these bf16 operands).
    want_best: return (nv, best_d, best_idx) — every row's nearest row of B under the canonical squared distance, lowest
    index on ties (the argmin of link mining).
    outsider_bound [n_rows]: the admission threshold the lists were collected under, if any (see snag_topk_rescore).
    norm_bound: an upper bound of ||a|| ||b|| the caller vouches for (saves the host round trip that measures it).
    lazy: no host synchronisation at all — the exhaustive completion is enqueued unconditionally (it reads the flagged
    count on the device and does nothing when it is zero) for at most the budgeted number of rows, and
    info[tag] holds the DEVICE counter ('flagged_dev') and 'budget_rows' for the caller to check later."""
    sfx = _suffix(A, B, "AB")
    info = LAST_TOPK_INFO if info is None else info
    _need(cand_idx, torch.int32, "cand_idx", 2)
    _need(cand_val, torch.float32, "cand_val", 2)
    n_rows = cand_idx.shape[0]
    dev = A.device
    st = current_stream()
    if outsider_bound is not None:
        _need(outsider_bound, torch.float32, "outsider_bound", 1)
        if outsider_bound.numel() < n_rows:
            raise ValueError("outsider_bound needs one entry per row")
    nv = torch.empty((n_rows,), dtype=torch.float32, device=dev)
    best_d = torch.empty((n_rows,), dtype=torch.float32, device=dev) if want_best else None
    best_i = torch.empty((n_rows,), dtype=torch.int32, device=dev) if want_best else None
    cap = n_rows
    flagged = torch.empty((cap,), dtype=torch.int32, device=dev)
    fcnt = torch.zeros((1,), dtype=torch.int32, device=dev)
    if margin is None:
        margin = tc_margin(A.shape[1], norm_bound) if norm_bound is not None else _error_scale(an, bn, A.shape[1])
    call("snag_topk_rescore" + sfx, ptr(A), ptr(B), A.shape[1], n_rows, ptr(an), ptr(bn), ptr(cand_idx), ptr(cand_val), k,
         TOPK_VERIFY_DELTA * margin, ptr(outsider_bound), ptr(nv), ptr(flagged), ptr(fcnt), cap,
         ptr(best_d), ptr(best_i), st)
    if lazy:
        budget_rows = int(min(cap, TOPK_EXHAUSTIVE_BUDGET // max(1, n_b * A.shape[1])))
        if budget_rows > 0:
            call("snag_topk_exhaustive" + sfx, ptr(A), ptr(B), A.shape[1], n_b, ptr(an), ptr(bn), ptr(flagged), ptr(fcnt), budget_rows,
                 k, ptr(nv), ptr(best_d), ptr(best_i), st)
        info[tag] = {"flagged_dev": fcnt, "budget_rows": budget_rows}
        return (nv, best_d, best_i) if want_best else nv
    n_flag = int(fcnt.item())
    info[tag] = {"flagged": n_flag, "unverified": 0}
    if n_flag:
        if float(n_flag) * n_b * A.shape[1] <= TOPK_EXHAUSTIVE_BUDGET:
            call("snag_topk_exhaustive" + sfx, ptr(A), ptr(B), A.shape[1], n_b, ptr(an), ptr(bn), ptr(flagged), ptr(fcnt), cap, k,
                 ptr(nv), ptr(best_d), ptr(best_i), st)
        else:
            info[tag]["unverified"] = n_flag
            import warnings
            warnings.warn(f"snag_b200: {n_flag} {tag} neighbourhoods could not be verified against the canonical arithmetic "
                          f"within the exhaustive budget (plateaus of near-equal similarities wider than {KT} - k); their "
                          f"CSLS means come from the tensor-core candidates and may differ from the reference in the last "
                          f"bits", RuntimeWarning, stacklevel=2)
    return (nv, best_d, best_i) if want_best else nv


def pair_score(X, Y, n: int, xn, yn, nv1, nv2, use_csls: bool, want_dot: bool = False):
    sfx = _suffix(X, Y)
    g = torch.empty((n,), dtype=torch.float32, device=X.device)
    s = torch.empty((n,), dtype=torch.float32, device=X.device) if want_dot else None
    call("snag_pair_score" + sfx, ptr(X), ptr(Y), X.shape[1], n, ptr(xn), ptr(yn), ptr(nv1), ptr(nv2), int(use_csls), ptr(g),
         ptr(s), current_stream())
    return (g, s) if want_dot else g


# Half-width of the rank sweep's deferral band, in units of the dot product s, as a multiple of tc_margin(): it has to
# cover (a) the tensor core's accumulation error against the fp64 index-order dot product (TC_DOT_ERR_PER_K above),
# (b) the roundings of the reference's fp32 chain (< 1e-6 in distance = 2.5e-7 in s) and (c) the roundings of the
# per-row / per-column thresholds (< 3e-7). A wider band only defers more elements to the canonical re-score
# (a few 1e4 of 1e12 at 1M x 1M).
RANK_BAND_EPS = 1.0


def _error_scale(xn: torch.Tensor, yn: torch.Tensor, dpad: int) -> float:
    """tc_margin for these operands: the measured bound scaled by the contraction width and by the largest
    ||x|| ||y|| present (align_ranks only lets nearly-unit rows through)."""
    norm = float(torch.sqrt(xn.max() * yn.max()).item())
    return tc_margin(dpad, norm)


def rank_band_eps(xn: torch.Tensor, yn: torch.Tensor, dpad: int) -> float:
    """Half-width of the deferral band (in s) for these operands — what eval_rank uses."""
    return RANK_BAND_EPS * _error_scale(xn, yn, dpad)


RANK_BAND_MIN_CAP = 1 << 20
RANK_BAND_PER_ROW = 16         # initial list capacity per evaluated row + column
RANK_BAND_MAX_CAP = 1 << 28    # beyond this many deferred elements (2 GB list) the in-kernel chain takes over


def eval_rank(X, Y, xn, yn, nv1, nv2, g_row, g_col, row_gid0: int, col_gid0: int, n1: int, n2: int, use_csls: bool,
              cnt_row: torch.Tensor, cnt_col: torch.Tensor, want_top3: bool = False, exact_chain: bool = False,
              norm_bound: float | None = None, lazy: bool = False, eps: float | None = None, canon: tuple | None = None,
              info: dict | None = None):
    """Rank counters of sweep 2, accumulated into cnt_row / cnt_col. Default: s-space sweep with a deferral band
    (snag_eval_rank_band) followed by the canonical re-score of the deferred elements (snag_band_rescore); a band list
    that overflows is retried with a larger list, and degenerate inputs (almost everything tied) fall back to the
    in-kernel fp32 chain (snag_eval_rank, `exact_chain=True`). Returns the per-list nearest-candidate lists
    ([n_lists, n1, 4] values, ids) when want_top3, else (None, None). info (default LAST_RANK_INFO) reports the attempt.
    eps: half-width of the band in s from the caller's error model (default: rank_band_eps of these bf16 operands).
    canon: the canonical rows (Xr, Yr) of the re-score when they are not X and Y (the fp32 rows of split operands).
    There is no chain on fp32 rows (its verdicts come from the tensor-core scores): their band list is clamped to
    RANK_BAND_MAX_CAP, and past it this raises.
    lazy: one attempt with the initial list capacity and no host synchronisation; info holds the DEVICE
    counter ('deferred_dev') and 'cap' — the caller must check deferred <= cap before trusting the counters."""
    _check_operand(X, "X")
    _check_operand(Y, "Y")
    Xc, Yc = (X, Y) if canon is None else canon
    sfx = _suffix(Xc, Yc)
    info = LAST_RANK_INFO if info is None else info
    _need(cnt_row, torch.int32, "cnt_row", 1)
    _need(cnt_col, torch.int32, "cnt_col", 1)
    t3v = t3i = None
    if want_top3:
        _, nch = sim_plan(n1, n2, X.shape[1])
        t3v = torch.empty((nch, n1, 4), dtype=torch.float32, device=X.device)
        t3i = torch.empty((nch, n1, 4), dtype=torch.int32, device=X.device)
    st = current_stream()
    if sfx and exact_chain:
        raise ValueError("the in-kernel chain ranks bf16 operands only")
    if not exact_chain:
        if eps is None:
            eps = RANK_BAND_EPS * (tc_margin(X.shape[1], norm_bound) if norm_bound is not None else _error_scale(xn, yn, X.shape[1]))
        cap = max(RANK_BAND_MIN_CAP, RANK_BAND_PER_ROW * (n1 + n2))

        def attempt(band, band_cnt, cap):
            with _SweepTimer("sim_kernel<EpiRank>", n1, n2):
                call("snag_eval_rank_band", ptr(X), ptr(Y), ptr(xn), ptr(yn), ptr(nv1), ptr(nv2), ptr(g_row), ptr(g_col),
                     row_gid0, col_gid0, n1, n2, X.shape[1], int(use_csls), eps, ptr(cnt_row), ptr(cnt_col),
                     ptr(t3v), ptr(t3i), ptr(band), ptr(band_cnt), cap, st)
            call("snag_band_rescore" + sfx, ptr(Xc), ptr(Yc), Xc.shape[1], ptr(xn), ptr(yn), ptr(nv1), ptr(nv2), ptr(g_row),
                 ptr(g_col), row_gid0, col_gid0, int(use_csls), ptr(band), ptr(band_cnt), cap, ptr(cnt_row), ptr(cnt_col), st)

        if lazy:
            band_cnt, cap = _band_retry(attempt, cap, (cnt_row, cnt_col), sync=False)
            info.clear()
            info.update(deferred_dev=band_cnt, cap=cap, mode="band", eps=eps)
            return t3v, t3i
        if sfx or cap <= RANK_BAND_MAX_CAP:
            deferred, cap = _band_retry(attempt, cap, (cnt_row, cnt_col), grow=8, max_cap=RANK_BAND_MAX_CAP, clamp=bool(sfx))
            if sfx:
                info.clear()
            info.update(deferred=deferred, cap=cap, mode="band", eps=eps)
            if deferred <= cap:
                return t3v, t3i
            if sfx:
                raise SnagError(f"{deferred} elements of the fp32 rank sweep are within the error bound of a ground-truth "
                                f"distance (nearly all ties): more than the deferral list can hold")
        # hopeless (nearly everything within the band: duplicated / constant embeddings): in-kernel chain with exact ties
    info.update(mode="chain")
    with _SweepTimer("sim_kernel<EpiRank>", n1, n2):
        call("snag_eval_rank", ptr(X), ptr(Y), ptr(xn), ptr(yn), ptr(nv1), ptr(nv2), ptr(g_row), ptr(g_col), row_gid0,
             col_gid0, n1, n2, X.shape[1], int(use_csls), ptr(cnt_row), ptr(cnt_col), ptr(t3v), ptr(t3i), st)
    if want_top3:                          # the chain kernel lists distances ascending; the merge expects x descending
        t3v = -t3v
        t3v[..., 3] = float("-inf")
        t3i[..., 3] = 0x7FFFFFFF
    return t3v, t3i


LAST_RANK_INFO: dict = {}


def pairs_dot(X, Y, rows: torch.Tensor, cols: torch.Tensor) -> torch.Tensor:
    """Canonical dot products X[rows[p]] . Y[cols[p]] (fp64 index-order accumulation, one rounding) of listed pairs of
    bf16 operands or fp32 rows."""
    sfx = _suffix(X, Y)
    _need(rows, torch.int32, "rows", 1)
    _need(cols, torch.int32, "cols", 1)
    if rows.numel() != cols.numel():
        raise ValueError("rows and cols must pair up")
    out = torch.empty((rows.numel(),), dtype=torch.float32, device=X.device)
    if rows.numel():
        call("snag_pairs_dot" + sfx, ptr(X), ptr(Y), X.shape[1], ptr(rows), ptr(cols), rows.numel(), ptr(out), current_stream())
    return out


def top4_merge(val: torch.Tensor, idx: torch.Tensor):
    """Merge per-list nearest-candidate lists [n_lists, n_rows, 4] (value descending, id ascending on ties) -> [n_rows, 4]."""
    _need(val, torch.float32, "val", 3)
    _need(idx, torch.int32, "idx", 3)
    n_lists, n_rows = val.shape[0], val.shape[1]
    oval = torch.empty((n_rows, 4), dtype=torch.float32, device=val.device)
    oidx = torch.empty((n_rows, 4), dtype=torch.int32, device=val.device)
    call("snag_top4_merge", ptr(val), ptr(idx), n_lists, n_rows, ptr(oval), ptr(oidx), current_stream())
    return oval, oidx


def top3_rescore(X, Y, xn, yn, nv1, nv2, use_csls: bool, cand: torch.Tensor):
    """Canonical distances of each row's candidate columns [n_rows, 4] (ids into Y), sorted ascending with the lower id
    first on ties: columns 0..2 are ret1..ret3 of the prediction file. Returns (val [n_rows, 4], idx [n_rows, 4])."""
    sfx = _suffix(X, Y)
    _need(cand, torch.int32, "cand", 2)
    n_rows = cand.shape[0]
    oval = torch.empty((n_rows, 4), dtype=torch.float32, device=cand.device)
    oidx = torch.empty((n_rows, 4), dtype=torch.int32, device=cand.device)
    call("snag_top3_rescore" + sfx, ptr(X), ptr(Y), X.shape[1], n_rows, ptr(xn), ptr(yn), ptr(nv1), ptr(nv2), int(use_csls),
         ptr(cand), ptr(oval), ptr(oidx), current_stream())
    return oval, oidx


def l1_distance(x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """fp32 [n1, n2] cityblock distances of fp32 rows (fp64 index-order accumulation, rounded once): --distance 1."""
    _need(x, torch.float32, "x", 2)
    _need(y, torch.float32, "y", 2)
    if x.shape[1] != y.shape[1]:
        raise ValueError("x and y must have the same width")
    out = torch.empty((x.shape[0], y.shape[0]), dtype=torch.float32, device=x.device)
    call("snag_l1_distance", ptr(x), ptr(y), x.shape[0], y.shape[0], x.shape[1], x.stride(0), y.stride(0), ptr(out),
         out.stride(0), current_stream())
    return out


def matrix_rank(dist: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    """(rank_l2r, rank_r2l) int32 [n] of the diagonal of a materialised square distance matrix (stable-sort positions)."""
    _need(dist, torch.float32, "distance", 2)
    n = dist.shape[0]
    if dist.shape[1] != n:
        raise ValueError("the distance matrix of n aligned pairs is square")
    cnt_row = torch.empty((n,), dtype=torch.int32, device=dist.device)
    cnt_col = torch.empty((n,), dtype=torch.int32, device=dist.device)
    call("snag_matrix_rank", ptr(dist), n, dist.stride(0), ptr(cnt_row), ptr(cnt_col), current_stream())
    return cnt_row, cnt_col


CSLS_MATRIX_K_MAX = 1024      # snag_csls_sim: k <= KT through the candidate-list passes, above that by radix selection


def csls_sim_matrix(sim: torch.Tensor, k: int, want_out: bool = True):
    """csls_sim on a materialised fp32 matrix: returns (out or None, nv1, nv2)."""
    _need(sim, torch.float32, "sim_mat", 2)
    n1, n2 = sim.shape
    if k > n1 or k > n2:
        raise RuntimeError("selected index k out of range")          # torch.topk's error in the reference
    if not 1 <= k <= CSLS_MATRIX_K_MAX:
        raise SnagError(f"csls_k={k} unsupported: at most {CSLS_MATRIX_K_MAX} neighbours on a materialised matrix")
    ws = torch.empty((_lib.load().snag_csls_workspace_bytes(n1, n2) // 4,), dtype=torch.float32, device=sim.device)
    nv1 = torch.empty((n1,), dtype=torch.float32, device=sim.device)
    nv2 = torch.empty((n2,), dtype=torch.float32, device=sim.device)
    out = torch.empty_like(sim) if want_out else None
    call("snag_csls_sim", ptr(sim), n1, n2, sim.stride(0), k, ptr(out), n2, ptr(nv1), ptr(nv2), ptr(ws), current_stream())
    return out, nv1, nv2


# ------------------------------------------------------------------------------------------------ ICL
def icl_side(X: torch.Tensor, Y: torch.Tensor, B: int, Bp: int, inv_tau: float, row0: int = 0, nx: int | None = None):
    """Row log-sum-exp and NLL of one side of the ICL loss for the anchors [row0, row0 + nx) of the batch (default: all).
    X [>= nx, Dpad] holds those anchors from its first row on, Y [2*Bp, Dpad] = [other side ; this side].
    Returns (lse, nll, pos) for the min(nx, B - row0) valid anchors."""
    _check_operand(X, "X")
    _check_operand(Y, "Y")
    nx = Bp if nx is None else int(nx)
    valid = max(0, min(nx, B - row0))
    if valid == 0:
        raise ValueError("no valid anchors in this shard")
    _, nch = sim_plan(nx, 2 * Bp, X.shape[1])
    part = torch.empty((nch, nx), dtype=torch.float32, device=X.device)
    pos = torch.empty((nx,), dtype=torch.float32, device=X.device)
    lse = torch.empty((valid,), dtype=torch.float32, device=X.device)
    nll = torch.empty((valid,), dtype=torch.float32, device=X.device)
    st = current_stream()
    with _SweepTimer("sim_kernel<EpiIclFwd>", nx, 2 * Bp, X.shape[1]):
        call("snag_icl_rowsum", ptr(X), ptr(Y), B, Bp, row0, nx, X.shape[1], inv_tau, ptr(part), ptr(pos), st)
    call("snag_icl_finalize", ptr(part), nch, valid, nx, ptr(pos), inv_tau, ptr(lse), ptr(nll), st)
    return lse, nll, pos


ICL_SYM_MAX_PROBLEMS = 16


def icl_fwd_sym(S3s, B: int, Bp: int, inv_tau: float, rank: int = 0, world: int = 1, all_reduce=None,
                esave=None, split: bool = False) -> torch.Tensor:
    """Forward statistics of icl_loss for several tables that share the batch, on half the Gram matrix of the stacked
    rows (snag_icl_fwd_sym): S3s[p] = [a ; b ; ...] as [>= 2 Bp, Dpad] bf16 (same Dpad). Returns fp32 [n_prob, 4, B] =
    (lse_a, nll_a, lse_b, nll_b) per table. With world > 1 this rank processes its contiguous share of the work units
    and `all_reduce(tensor) -> tensor` (sum over the ranks) combines the partial sums before the logarithm.
    esave: optional list (one entry per table, None to skip) of bf16 [2 Bp, 2 Bp] buffers that receive E of every computed
    element for icl_g_from_e (single rank only: the buffer must see all work units).
    split: S3s are the split stacks of the fp32 loss route ([3 Bp, 5 Dpad], snag_icl_fwd_sym_split; no esave)."""
    import ctypes
    n_prob = len(S3s)
    if not 1 <= n_prob <= ICL_SYM_MAX_PROBLEMS:
        raise ValueError(f"1..{ICL_SYM_MAX_PROBLEMS} tables per launch")
    if split and esave is not None:
        raise ValueError("esave is not available for split stacks: a bf16 E would cap dL/dlogits at 2^-9 relative")
    dpad = S3s[0].shape[1]
    for t in S3s:
        _check_operand(t, "S3")
        if t.shape[0] < 2 * Bp or t.shape[1] != dpad:
            raise ValueError("every stacked operand must be [>= 2 * Bp, Dpad] with the same Dpad")
    dev = S3s[0].device
    sizes = (ctypes.c_int64 * 3)()
    call("snag_icl_fwd_sym_plan", n_prob, B, Bp, sizes)
    units, rp, cp = int(sizes[0]), int(sizes[1]), int(sizes[2])
    u0, u1 = units * rank // world, units * (rank + 1) // world
    rowpart = torch.empty((n_prob, rp), dtype=torch.float32, device=dev)
    colpart = torch.empty((n_prob, cp), dtype=torch.float32, device=dev)
    # total and pos travel in one buffer so that a sharded step needs a single all-reduce
    buf = torch.zeros((n_prob * 3 * Bp,), dtype=torch.float32, device=dev) if world > 1 else \
        torch.empty((n_prob * 3 * Bp,), dtype=torch.float32, device=dev)
    total, pos = buf[:n_prob * 2 * Bp], buf[n_prob * 2 * Bp:]
    arr = lambda ts: (ctypes.c_void_p * n_prob)(*[None if t is None else t.data_ptr() for t in ts])
    es = None
    if esave is not None and any(t is not None for t in esave):
        if world != 1 or len(esave) != n_prob:
            raise ValueError("esave needs one entry per table and an unsharded launch")
        for t in esave:
            if t is not None and (t.dtype != torch.bfloat16 or tuple(t.shape) != (2 * Bp, 2 * Bp) or not t.is_contiguous()):
                raise ValueError("esave buffers must be contiguous bf16 [2 Bp, 2 Bp]")
        es = arr(esave)
    tiles = (2 * Bp // 256) ** 2 + 2 * Bp // 256            # per table: the staircase of 128-row blocks x 256-column tiles
    share = (u1 - u0) / max(1, units)
    if split:
        if dpad % 320:
            raise ValueError("split stacks are [3 Bp, 5 Dpad] with Dpad a multiple of 64")
        with _SweepTimer("icl_fwd_sym_split_kernel", int(n_prob * tiles * share) * 128, 256, dpad // 5 * 3):
            call("snag_icl_fwd_sym_split", n_prob, arr(S3s), arr([rowpart[i] for i in range(n_prob)]),
                 arr([colpart[i] for i in range(n_prob)]), ptr(pos), B, Bp, dpad // 5, float(inv_tau), u0, u1, ptr(total),
                 current_stream())
    else:
        with _SweepTimer("icl_fwd_sym_kernel", int(n_prob * tiles * share) * 128, 256, dpad):
            call("snag_icl_fwd_sym", n_prob, arr(S3s), arr([rowpart[i] for i in range(n_prob)]),
                 arr([colpart[i] for i in range(n_prob)]), ptr(pos), B, Bp, dpad, float(inv_tau), u0, u1, ptr(total), es,
                 current_stream())
    if world > 1:
        buf = all_reduce(buf)
        total, pos = buf[:n_prob * 2 * Bp], buf[n_prob * 2 * Bp:]
    out = torch.empty((n_prob, 4, B), dtype=torch.float32, device=dev)
    call("snag_icl_sym_finalize", ptr(total), ptr(pos), n_prob, B, Bp, float(inv_tau), ptr(out), current_stream())
    return out


def icl_g_from_e(E: torch.Tensor, side: int, B: int, Bp: int, cr_this: torch.Tensor, cr_other: torch.Tensor,
                 diag: torch.Tensor, inv_tau: float) -> torch.Tensor:
    """dL/dlogits of one side (bf16 [Bp, 2 Bp], what icl_bwd_logits returns for all anchors) formed from the E the
    half-Gram forward saved (snag_icl_g_from_e): a bandwidth kernel instead of a recomputation of the logits.
    diag [B]: the cross-diagonal values G[i, i] = (g_a expm1(-nll_a) + g_b expm1(-nll_b)) / tau (see the header)."""
    if E.dtype != torch.bfloat16 or tuple(E.shape) != (2 * Bp, 2 * Bp) or not E.is_contiguous():
        raise ValueError("E must be contiguous bf16 [2 Bp, 2 Bp]")
    for t, nm in ((cr_this, "cr_this"), (cr_other, "cr_other"), (diag, "diag")):
        _need(t, torch.float32, nm, 1)
        if t.numel() < B:
            raise ValueError(f"{nm} needs at least B entries")
    G = torch.empty((Bp, 2 * Bp), dtype=torch.bfloat16, device=E.device)
    call("snag_icl_g_from_e", ptr(E), int(side), B, Bp, ptr(cr_this), ptr(cr_other), ptr(diag), float(inv_tau), ptr(G),
         current_stream())
    return G


def icl_bwd_logits(X: torch.Tensor, Y: torch.Tensor, B: int, Bp: int, inv_tau: float, cr: torch.Tensor,
                   cc: torch.Tensor, dg: torch.Tensor, row0: int = 0, nx: int | None = None,
                   self_cols: bool = True, ebar: float = 0.0) -> torch.Tensor:
    """dL/dlogits of one ICL side as bf16 [nx, 2*Bp] for the anchors [row0, row0 + nx) of the batch (default: all Bp
    rows of the side); see snag_icl_bwd_logits."""
    _check_operand(X, "X")
    _check_operand(Y, "Y")
    nx = Bp if nx is None else int(nx)
    for t, nm in ((cr, "cr"), (cc, "cc"), (dg, "dg")):
        _need(t, torch.float32, nm, 1)
        if t.numel() < B:
            raise ValueError(f"{nm} needs at least B entries")
    G = torch.empty((nx, 2 * Bp), dtype=torch.bfloat16, device=X.device)
    with _SweepTimer("sim_kernel<EpiIclBwd>", nx, 2 * Bp, X.shape[1]):
        call("snag_icl_bwd_logits", ptr(X), ptr(Y), B, Bp, row0, nx, X.shape[1], inv_tau, ptr(cr), ptr(cc), ptr(dg), ptr(G),
             int(self_cols), float(ebar), current_stream())
    return G


MANY_MAX = 16                 # problems per batched launch (kernel-parameter space)


def _carr(ctype, values):
    return (ctype * len(values))(*values)


def icl_stack_prep(embs, idx_l: torch.Tensor, idx_r: torch.Tensor, Bp: int, normalize: bool = True):
    """Stacked bf16 operands of several icl_loss calls that share one batch, ONE launch per 16 tables: for each fp32
    table emb [N, D] returns S3 = [z[idx_l] ; z[idx_r] ; z[idx_l]] as [3 Bp, Dpad] bf16 (z = F.normalize(emb) when
    `normalize`), every part zero padded to Bp rows and Dpad = ceil(D / 64) * 64 columns."""
    import ctypes as C
    _need(idx_l, torch.int64, "idx_l", 1)
    _need(idx_r, torch.int64, "idx_r", 1)
    B = idx_l.numel()
    if idx_r.numel() != B or B < 1 or Bp < B or Bp % 256:
        raise ValueError("idx_l / idx_r must pair up and Bp must be a multiple of 256 >= B")
    outs = []
    for e in embs:
        _need(e, torch.float32, "emb", 2)
        outs.append(torch.empty((3 * Bp, round_up(e.shape[1], 64)), dtype=torch.bfloat16, device=e.device))
    for i in range(0, len(embs), MANY_MAX):
        es, os_ = embs[i:i + MANY_MAX], outs[i:i + MANY_MAX]
        call("snag_icl_stack_prep", len(es), _carr(C.c_void_p, [e.data_ptr() for e in es]),
             _carr(C.c_int64, [e.stride(0) for e in es]), _carr(C.c_int32, [e.shape[1] for e in es]),
             _carr(C.c_void_p, [t.data_ptr() for t in os_]), _carr(C.c_int32, [t.shape[1] for t in os_]),
             ptr(idx_l), ptr(idx_r), B, Bp, int(normalize), current_stream())
    return outs


def normalize_bwd_scatter_many(embs, idx_l: torch.Tensor, idx_r: torch.Tensor, dz_pairs, dembs, normalize: bool = True):
    """normalize_bwd_scatter for both sides of several tables in ONE launch per 16 tables: dembs[p][idx_l[r]] +=
    backward of F.normalize(embs[p][idx_l[r]]) applied to dz_pairs[p][0][r] (and idx_r / dz_pairs[p][1] likewise);
    every dz is [>= n, >= D] or [n_parts, >= n, >= D] with n = idx_l.numel()."""
    import ctypes as C
    n = idx_l.numel()
    for i in range(0, len(embs), MANY_MAX):
        sl = slice(i, i + MANY_MAX)
        es, ds, gs = embs[sl], dembs[sl], dz_pairs[sl]
        ld_dz, n_parts, pstride = [], [], []
        for e, d, (ga, gb) in zip(es, ds, gs):
            _need(e, torch.float32, "emb", 2)
            _need(d, torch.float32, "demb", 2)
            if ga.shape != gb.shape or ga.stride() != gb.stride() or ga.dtype != torch.float32 or ga.stride(-1) != 1:
                raise ValueError("the two sides' gradients must share shape and layout (fp32, contiguous rows)")
            if ga.shape[-2] < n or ga.shape[-1] < e.shape[1] or d.shape != e.shape:
                raise ValueError("normalize_bwd_scatter_many: shape mismatch")
            ld_dz.append(ga.stride(-2))
            n_parts.append(1 if ga.dim() == 2 else ga.shape[0])
            pstride.append(0 if ga.dim() == 2 else ga.stride(0))
        call("snag_normalize_bwd_scatter_many", len(es), _carr(C.c_void_p, [e.data_ptr() for e in es]),
             _carr(C.c_int64, [e.stride(0) for e in es]), _carr(C.c_int32, [e.shape[1] for e in es]),
             _carr(C.c_void_p, [g[0].data_ptr() for g in gs]), _carr(C.c_void_p, [g[1].data_ptr() for g in gs]),
             _carr(C.c_int64, ld_dz), _carr(C.c_int32, n_parts), _carr(C.c_int64, pstride),
             _carr(C.c_void_p, [d.data_ptr() for d in ds]), _carr(C.c_int64, [d.stride(0) for d in ds]),
             ptr(idx_l), ptr(idx_r), n, int(normalize), current_stream())


FUSED_BWD_MAX_DPAD = 320      # dZ accumulator (Dpad fp32 columns) + logits stages + P buffers must fit the 512 TMEM columns
FUSED_BWD_MAX_PROBLEMS = 16


def icl_bwd_fused(S3s, cras, crbs, dgs, B: int, Bp: int, inv_tau: float, row0: int = 0, nx: int | None = None):
    """Fused backward of icl_loss w.r.t. the normalised rows for Dpad <= 320 (snag_icl_bwd_fused): for each problem p
    (stacked operand S3s[p] = [a ; b ; a] as [3 Bp, Dpad] bf16, row coefficients cras[p] / crbs[p] and diagonal term
    dgs[p], all [>= B] fp32) returns (dz_a, dz_b), each [nsplit, nx, Dpad] fp32: the partial gradients of the anchors
    [row0, row0 + nx) of side a / b over the column splits (sum over dim 0 = dL/dz). No [B, 2B] matrix touches HBM."""
    import ctypes
    n_prob = len(S3s)
    if not 1 <= n_prob <= FUSED_BWD_MAX_PROBLEMS or not (len(cras) == len(crbs) == len(dgs) == n_prob):
        raise ValueError(f"1..{FUSED_BWD_MAX_PROBLEMS} problems with one coefficient set each")
    nx = Bp if nx is None else int(nx)
    if row0 % 128 or nx % 128 or nx < 128 or row0 + nx > Bp:
        raise ValueError("anchor range must be whole blocks of 128 rows inside [0, Bp)")
    dpad = S3s[0].shape[1]
    for t in S3s:
        _check_operand(t, "S3")
        if tuple(t.shape) != (3 * Bp, dpad):
            raise ValueError("every stacked operand must be [3 * Bp, Dpad] with the same Dpad")
    if dpad > FUSED_BWD_MAX_DPAD:
        raise SnagError(f"fused ICL backward supports Dpad <= {FUSED_BWD_MAX_DPAD}, got {dpad}")
    for lst, nm in ((cras, "cr_a"), (crbs, "cr_b"), (dgs, "dg")):
        for t in lst:
            _need(t, torch.float32, nm, 1)
            if t.numel() < B:
                raise ValueError(f"{nm} needs at least B entries")
    dev = S3s[0].device
    rbs = nx // 128
    nsplit = int(_lib.load().snag_icl_bwd_fused_splits(n_prob, B, Bp, rbs))
    # one allocation for all partial outputs: [problem][side][split][nx][Dpad]
    out = torch.empty((n_prob, 2, nsplit, nx, dpad), dtype=torch.float32, device=dev)
    arr = lambda ts: (ctypes.c_void_p * n_prob)(*[t.data_ptr() for t in ts])
    with _SweepTimer("icl_bwd_fused_kernel", 2 * n_prob * nx, 2 * Bp, 2 * dpad):      # two MMAs per logits element
        call("snag_icl_bwd_fused", n_prob, arr(S3s), arr(cras), arr(crbs), arr(dgs), arr([out[i, 0] for i in range(n_prob)]),
             arr([out[i, 1] for i in range(n_prob)]), B, Bp, row0 // 128, rbs, dpad, float(inv_tau), nsplit, nx * dpad,
             current_stream())
    return [(out[i, 0], out[i, 1]) for i in range(n_prob)]


def contract(P: torch.Tensor, Q: torch.Tensor, n1: int, n2: int) -> torch.Tensor:
    """fp32 [n1, n2] = P[:n1] . Q[:n2]^T for bf16 operands sharing the (multiple-of-64) contraction width — the
    gradient GEMMs of the loss layer run on the same tcgen05 mainloop as the similarity sweeps."""
    return sim_write(P, Q, None, None, n1, n2, 0)


def grad_contract_rows(G: torch.Tensor, Yrows: torch.Tensor, n_rows: int, d: int, keep_parts: bool = False) -> torch.Tensor:
    """fp32 [n_rows, d] = G[:n_rows] . Yrows[:, :d] for bf16 G [>= n_rows, K] and Yrows [K, Dpad] (contiguous rows, Dpad a
    multiple of 64, K a multiple of 64): grad_contract without the transposed copy of the stacked embeddings — the tensor
    cores read Yrows' tiles MN-major (snag_sim_write_t_mn)."""
    _check_operand(G, "G")
    _check_operand(Yrows, "Yrows")
    k = G.shape[1]
    if Yrows.shape[0] != k or Yrows.shape[1] < d:
        raise ValueError("Yrows must be [K, >= d] with K = G's contraction width")
    ks = int(_lib.load().snag_sim_write_t_splits(d, n_rows, k))
    part = torch.empty((ks, n_rows, d), dtype=torch.float32, device=G.device)
    with _SweepTimer("sim_kernel<EpiWrite>", d, n_rows, k):
        call("snag_sim_write_t_mn", ptr(Yrows), Yrows.shape[1], ptr(G), d, n_rows, k, ks, ptr(part), d, n_rows * d,
             current_stream())
    if keep_parts:
        return part
    return part[0] if ks == 1 else part.sum(0)


def grad_contract(G: torch.Tensor, YT: torch.Tensor, n_rows: int, d: int, keep_parts: bool = False) -> torch.Tensor:
    """fp32 [n_rows, d] = G[:n_rows] . YT[:d]^T for bf16 G [>= n_rows, K] and YT [>= d, K] (K a multiple of 64): the
    loss's gradient GEMMs dX = dL/dlogits . [other ; this]. Runs with the d rows of YT as the X operand, the output
    written transposed and the long contraction split over the SMs (see snag_sim_write_t). keep_parts: return the
    split-K partial products [ks, n_rows, d] instead of their sum (normalize_bwd_scatter adds them while it reads)."""
    _check_operand(G, "G")
    _check_operand(YT, "YT")
    if G.shape[1] != YT.shape[1]:
        raise ValueError("contraction widths differ")
    k = G.shape[1]
    ks = int(_lib.load().snag_sim_write_t_splits(d, n_rows, k))
    part = torch.empty((ks, n_rows, d), dtype=torch.float32, device=G.device)
    with _SweepTimer("sim_kernel<EpiWrite>", d, n_rows, k):
        call("snag_sim_write_t", ptr(YT), ptr(G), d, n_rows, k, ks, ptr(part), d, n_rows * d, current_stream())
    if keep_parts:                       # [ks, n_rows, d]: the consumer adds the split-K partial sums itself
        return part
    return part[0] if ks == 1 else part.sum(0)


# ------------------------------------------------------------------------------------------------ noise
def noise_mask(x: torch.Tensor, mean: torch.Tensor, std: torch.Tensor, noise_ratio: float, mask_ratio: float, *,
               out: torch.Tensor | None = None, mask: torch.Tensor | None = None, zsel: torch.Tensor | None = None,
               seed: int = 0, row0: int = 0) -> torch.Tensor:
    _need(x, torch.float32, "x", 2)
    _need(mean, torch.float32, "mean", 1)
    _need(std, torch.float32, "std", 1)
    if x.shape[1] % 4:
        # the kernel moves one float4 per thread; a feature width that is not a multiple of 4 (e.g. the attribute matrix of
        # a dataset with fewer than 1000 distinct attributes, src/data.py:507) is zero padded for the call and cut back
        pad = 4 - x.shape[1] % 4
        P = torch.nn.functional.pad
        res = noise_mask(P(x, (0, pad)), P(mean, (0, pad)), P(std, (0, pad)), noise_ratio, mask_ratio, mask=mask,
                         zsel=None if zsel is None else P(zsel, (0, pad)), seed=seed, row0=row0)[:, :x.shape[1]]
        if out is None:
            return res.contiguous()
        out.copy_(res)
        return out
    if out is None:
        out = torch.empty_like(x)
    _need(out, torch.float32, "out", 2)
    selpos = None
    if mask is not None:
        _need(mask, torch.uint8, "mask", 1)
    if zsel is not None:
        if mask is None:
            raise ValueError("zsel needs the row mask it was drawn for")
        _need(zsel, torch.float32, "zsel", 2)
        selpos = (torch.cumsum(mask.to(torch.int32), 0, dtype=torch.int32) - 1).contiguous()
    if mask is None:
        # the Bernoulli row selection once per row (N Philox draws) rather than once per float4 inside the mask kernel:
        # same counter, same stream, so the output is the same function of (seed, row, column)
        mask = philox_rowmask(x.shape[0], noise_ratio, seed, x.device, row0)
    keep = float(1.0 - mask_ratio)
    call("snag_noise_mask", ptr(x), ptr(out), ptr(mean), ptr(std), ptr(mask), ptr(zsel), ptr(selpos), x.shape[0],
         x.shape[1], x.stride(0), out.stride(0), float(noise_ratio), keep, float(mask_ratio), int(seed), int(row0),
         current_stream())
    return out


def philox_rowmask(n: int, ratio: float, seed: int, device, row0: int = 0) -> torch.Tensor:
    mask = torch.empty((n,), dtype=torch.uint8, device=device)
    call("snag_philox_rowmask", ptr(mask), n, float(ratio), int(seed), int(row0), current_stream())
    return mask


def gauss_fill(mean: torch.Tensor, std: torch.Tensor, n: int, seed: int, row0: int = 0) -> torch.Tensor:
    _need(mean, torch.float32, "mean", 1)
    _need(std, torch.float32, "std", 1)
    if mean.numel() % 4:                                   # float4 kernel: pad the width for the call (see noise_mask)
        pad = 4 - mean.numel() % 4
        P = torch.nn.functional.pad
        return gauss_fill(P(mean, (0, pad)), P(std, (0, pad)), n, seed, row0)[:, :mean.numel()].contiguous()
    out = torch.empty((n, mean.numel()), dtype=torch.float32, device=mean.device)
    call("snag_gauss_fill", ptr(out), ptr(mean), ptr(std), n, mean.numel(), out.stride(0), int(seed), int(row0),
         current_stream())
    return out


def col_mean_std(x: torch.Tensor, valid: torch.Tensor | None = None) -> tuple[torch.Tensor, torch.Tensor]:
    _need(x, torch.float32, "x", 2)
    if valid is not None:
        _need(valid, torch.uint8, "valid", 1)
    f = x.shape[1]
    mean = torch.empty((f,), dtype=torch.float32, device=x.device)
    std = torch.empty((f,), dtype=torch.float32, device=x.device)
    ws = torch.empty((2 * f + 1,), dtype=torch.float64, device=x.device)
    call("snag_col_mean_std", ptr(x), ptr(valid), x.shape[0], f, x.stride(0), ptr(mean), ptr(std), ptr(ws),
         current_stream())
    return mean, std


def rowblend_fwd(e: torch.Tensor, noise: torch.Tensor, mask: torch.Tensor, a: float, c: float) -> torch.Tensor:
    _need(e, torch.float32, "e", 2)
    _need(noise, torch.float32, "noise", 2)
    _need(mask, torch.uint8, "mask", 1)
    out = torch.empty_like(e)
    call("snag_rowblend_fwd", ptr(e), ptr(noise), ptr(mask), ptr(out), e.shape[0], e.shape[1], a, c, current_stream())
    return out


def rowblend_bwd(g: torch.Tensor, mask: torch.Tensor, a: float) -> torch.Tensor:
    _need(g, torch.float32, "g", 2)
    gin = torch.empty_like(g)
    call("snag_rowblend_bwd", ptr(g), ptr(mask), ptr(gin), g.shape[0], g.shape[1], a, current_stream())
    return gin
