"""Kernel backend of the fp32 loss route (icl_loss with precision "fp32", loss.TRAIN_PRECISION): the entry points
loss._IclMany calls, over a three-term bf16 split of the UNROUNDED normalised rows instead of their bf16 rounding.

Every table is carried as one split stack, a bf16 tensor [3 Bp, 5 Dpad] (snag_icl_stack_prep_split): row r of
[a ; b ; a] laid out [m | h | h | m | h] with h = bf16(z), m = bf16(z - h). Its side-0 window (columns [0, 3 Dpad)) is
[m | h | h] and its side-1 window (columns [2 Dpad, 5 Dpad)) is [h | m | h], so a contraction of a side-0 row with a
side-1 row over 3 Dpad forms m_i h_j + h_i m_j + h_i h_j — symmetric in (i, j), so the half-Gram forward, its staircase
and its sums stay valid. The stack is a plain tensor (autograd saves it) and _IclMany slices its rows exactly as it
slices a bf16 stack [3 Bp, Dpad]; the windows are taken here, by pointer and row stride, without copies.

Backward: dL/dlogits G is formed in fp32 from the split logits and written as G3 = [G_h | G_h | G_m] ([nx, 6 Bp]); the
gradient GEMM contracts it over K = 6 Bp with the K-stacked rows [Y_h ; Y_m ; Y_h] of the side-1 window ([6 Bp, Dpad],
one bandwidth copy per side: 6 Bp Dpad bf16, 0.36 GB at B = 16 384, D = 1800), i.e. G_h Y_h + G_h Y_m + G_m Y_h.

Deliberately absent: icl_bwd_fused (its tensor memory holds one accumulator of Dpad <= 320, not 3 Dpad) and
icl_g_from_e (a bf16 E caps G at 2^-9 relative), so _IclMany takes the two-kernel backward for every width.

Error model (per logit, unit rows): |s_tc - z_i.z_j| <= fp32.tc_margin(Dpad) (the measured accumulation error of the
tensor cores on split operands, the proven split term 3 * 2^-16 and half an fp32 ulp); per element of G: 2^-16 |G| from
the two-term split of G plus the dropped G_m Y_m, against 2^-8 |G| for the bf16 route."""
from __future__ import annotations

import torch

from . import ops
from ._lib import call, current_stream, ptr
from .ops import _SweepTimer, _carr, _check_operand, _need, round_up, sim_plan

normalize_bwd_scatter = ops.normalize_bwd_scatter
normalize_bwd_scatter_many = ops.normalize_bwd_scatter_many


def _dpad(S: torch.Tensor) -> int:
    _check_operand(S, "split stack")
    if S.shape[1] % 320:
        raise ValueError(f"split stacks are [rows, 5 Dpad] with Dpad a multiple of 64, got width {S.shape[1]}")
    return S.shape[1] // 5


def _side1(S: torch.Tensor, dpad: int) -> int:
    """device address of the side-1 window of S's first row ([h | m | h], 2 Dpad columns in)"""
    return S.data_ptr() + 2 * dpad * S.element_size()


def icl_stack_prep(embs, idx_l: torch.Tensor, idx_r: torch.Tensor, Bp: int, normalize: bool = True):
    """Split stacks [3 Bp, 5 Dpad] bf16 of several tables that share the batch, ONE launch per 16 tables
    (snag_icl_stack_prep_split): h is bit for bit ops.icl_stack_prep's output, m bit for bit fp32.prep's."""
    import ctypes as C
    _need(idx_l, torch.int64, "idx_l", 1)
    _need(idx_r, torch.int64, "idx_r", 1)
    B = idx_l.numel()
    if idx_r.numel() != B or B < 1 or Bp < B or Bp % 256:
        raise ValueError("idx_l / idx_r must pair up and Bp must be a multiple of 256 >= B")
    outs, dpads = [], []
    for e in embs:
        _need(e, torch.float32, "emb", 2)
        dpads.append(round_up(e.shape[1], 64))
        outs.append(torch.empty((3 * Bp, 5 * dpads[-1]), dtype=torch.bfloat16, device=e.device))
    for i in range(0, len(embs), ops.MANY_MAX):
        es, os_, ds = embs[i:i + ops.MANY_MAX], outs[i:i + ops.MANY_MAX], dpads[i:i + ops.MANY_MAX]
        call("snag_icl_stack_prep_split", len(es), _carr(C.c_void_p, [e.data_ptr() for e in es]),
             _carr(C.c_int64, [e.stride(0) for e in es]), _carr(C.c_int32, [e.shape[1] for e in es]),
             _carr(C.c_void_p, [t.data_ptr() for t in os_]), _carr(C.c_int32, ds),
             ptr(idx_l), ptr(idx_r), B, Bp, int(normalize), current_stream())
    return outs


def icl_fwd_sym(S5s, B: int, Bp: int, inv_tau: float, rank: int = 0, world: int = 1, all_reduce=None) -> torch.Tensor:
    """ops.icl_fwd_sym on split stacks: fp32 [n_prob, 4, B] = (lse_a, nll_a, lse_b, nll_b) per table."""
    return ops.icl_fwd_sym(S5s, B, Bp, inv_tau, rank, world, all_reduce, split=True)


def icl_side(X: torch.Tensor, Y: torch.Tensor, B: int, Bp: int, inv_tau: float, row0: int = 0, nx: int | None = None):
    """ops.icl_side on split stacks: X = the anchors' rows, Y = the rows of [other ; this] (both [.., 5 Dpad]);
    the sweep contracts X's side-0 window with Y's side-1 window (snag_icl_rowsum_split)."""
    dpad = _dpad(X)
    if _dpad(Y) != dpad:
        raise ValueError("X and Y must be split stacks of the same table")
    nx = Bp if nx is None else int(nx)
    valid = max(0, min(nx, B - row0))
    if valid == 0:
        raise ValueError("no valid anchors in this shard")
    _, nch = sim_plan(nx, 2 * Bp, 3 * dpad)
    part = torch.empty((nch, nx), dtype=torch.float32, device=X.device)
    pos = torch.empty((nx,), dtype=torch.float32, device=X.device)
    lse = torch.empty((valid,), dtype=torch.float32, device=X.device)
    nll = torch.empty((valid,), dtype=torch.float32, device=X.device)
    st = current_stream()
    with _SweepTimer("sim_kernel<EpiIclFwd>", nx, 2 * Bp, 3 * dpad):
        call("snag_icl_rowsum_split", ptr(X), _side1(Y, dpad), B, Bp, row0, nx, dpad, inv_tau, ptr(part), ptr(pos), st)
    call("snag_icl_finalize", ptr(part), nch, valid, nx, ptr(pos), inv_tau, ptr(lse), ptr(nll), st)
    return lse, nll, pos


def icl_bwd_logits(X: torch.Tensor, Y: torch.Tensor, B: int, Bp: int, inv_tau: float, cr: torch.Tensor,
                   cc: torch.Tensor, dg: torch.Tensor, row0: int = 0, nx: int | None = None) -> torch.Tensor:
    """ops.icl_bwd_logits on split stacks (windows as icl_side): G3 = [G_h | G_h | G_m] bf16 [nx, 6 Bp]
    (snag_icl_bwd_logits_split)."""
    dpad = _dpad(X)
    if _dpad(Y) != dpad:
        raise ValueError("X and Y must be split stacks of the same table")
    nx = Bp if nx is None else int(nx)
    for t, nm in ((cr, "cr"), (cc, "cc"), (dg, "dg")):
        _need(t, torch.float32, nm, 1)
        if t.numel() < B:
            raise ValueError(f"{nm} needs at least B entries")
    G3 = torch.empty((nx, 6 * Bp), dtype=torch.bfloat16, device=X.device)
    with _SweepTimer("sim_kernel<EpiIclBwdSplit>", nx, 2 * Bp, 3 * dpad):
        call("snag_icl_bwd_logits_split", ptr(X), _side1(Y, dpad), B, Bp, row0, nx, dpad, inv_tau, ptr(cr), ptr(cc),
             ptr(dg), ptr(G3), current_stream())
    return G3


def k_stack(Yrows: torch.Tensor) -> torch.Tensor:
    """[Y_h ; Y_m ; Y_h] ([3 n, Dpad] bf16) of split-stack rows Yrows [n, 5 Dpad]: their side-1 window [h | m | h] with
    the three column blocks stacked along the rows (one bandwidth copy)."""
    dpad = _dpad(Yrows)
    n = Yrows.shape[0]
    return Yrows[:, 2 * dpad:].view(n, 3, dpad).transpose(0, 1).reshape(3 * n, dpad)


def grad_contract_rows(G3: torch.Tensor, Yrows: torch.Tensor, n_rows: int, d: int, keep_parts: bool = False) -> torch.Tensor:
    """fp32 [n_rows, d] = G_h Y_h + G_h Y_m + G_m Y_h for G3 from icl_bwd_logits and the split-stack rows Yrows
    [2 Bp, 5 Dpad] of [other ; this]: one ops.grad_contract_rows over K = 6 Bp."""
    Y3 = k_stack(Yrows)
    if G3.shape[1] != Y3.shape[0]:
        raise ValueError("G3 must be [n, 6 Bp] for Yrows [2 Bp, 5 Dpad]")
    return ops.grad_contract_rows(G3, Y3, n_rows, d, keep_parts=keep_parts)
