"""ICL / IAL in-batch contrastive losses and the uncertainty-weighting layer — host-side mirror of
SNAG_MMEA/model/SNAG_loss.py (same class names, constructor arguments, forward signatures and parameter
names, so `from snag_b200.loss import CustomMultiLossLayer, icl_loss, ial_loss` replaces the reference import
in model/SNAG.py:12 unchanged).

icl_loss: the four B x B similarity contractions, the -1e9 self-mask, the concatenation and the soft-label
cross entropy of model/SNAG_loss.py:98-126 are one fused tcgen05 sweep per side (row log-sum-exp in the
epilogue, no B x 2B matrix in HBM); the backward recomputes the logits tile by tile, writes dL/dlogits in bf16
and contracts it with the stacked embeddings on the same mainloop. Gather, normalisation, the per-pair weight
min(w[l], w[r]) and the final means stay ordinary torch autograd, so gradients reach `emb` and `weight_norm`
exactly as in the reference (model/SNAG_loss.py:51,66-69).

ial_loss (constructed but never called by SNAG — model/SNAG.py:53; live caller model/MCLEA.py:128-139): the KL between
the softmaxes of the two sets of logits is evaluated row-wise from the same fused sweeps as icl_loss — row log-sum-exps
of both sets, the target probabilities written once in bf16 and contracted with the stacked embeddings — so no fp32
[B, 2B] matrix exists; `norm=False` and unreduced outputs (no caller in the reference) are refused.
"""
from __future__ import annotations

import copy
import os

import numpy as np
import torch
from torch import nn

from . import ops


def cosine_sim(im, s):
    """model/SNAG_loss.py:7-10 (helper kept for interface parity; unused by the forwards, as in the reference)."""
    return _Contract.apply(im, s)


class CustomMultiLossLayer(nn.Module):
    """model/SNAG_loss.py:12-29 — sum_i exp(-s_i) * L_i + s_i over at most `loss_num` scalars. Stays in torch
    (six scalars). The parameter keeps the name `log_vars`: src/utils.py:46-54 gives `multi_loss_layer*`
    parameters their own learning rate by name."""

    def __init__(self, loss_num):
        super().__init__()
        self.loss_num = loss_num
        self.log_vars = nn.Parameter(torch.zeros(self.loss_num, ), requires_grad=True)

    def forward(self, loss_list):
        """sum_i exp(-s_i) * L_i + s_i over the first len(loss_list) entries; an entry may be the int 0 of an absent
        modality (model/SNAG.py:147-160), which still contributes its s_i."""
        k = len(loss_list)
        assert k <= self.loss_num
        if k == 0:
            return 0
        lv = self.log_vars
        # numeric entries become device scalars through a fill (no host -> device copy: the step stays graph capturable)
        terms = torch.stack([l.to(lv.dtype) if isinstance(l, torch.Tensor) else lv.new_full((), float(l)) for l in loss_list])
        return (torch.exp(-self.log_vars[:k]) * terms + self.log_vars[:k]).sum()


class AutomaticWeightedLoss(nn.Module):
    """model/Tool_model.py:14-37 — sum_i 0.5 / p_i^2 * L_i + log(1 + p_i^2) with learnable `params` (ones). SNAG builds
    one with num=7 as `multi_loss_layer_2` (model/SNAG.py:49); its name puts it in the 5x-lr, no-decay optimiser group
    (src/utils.py:46-54) and its `params` entry is part of the state dict whether or not --awloss is set."""

    def __init__(self, num=2, args=None):
        super().__init__()
        learn = args is None or args.use_awl
        self.params = nn.Parameter(torch.ones(num), requires_grad=bool(learn))

    def forward(self, *x):
        loss_sum = 0
        for i, loss in enumerate(x):
            loss_sum += 0.5 / (self.params[i] ** 2) * loss + torch.log(1 + self.params[i] ** 2)
        return loss_sum


# The kernels evaluate E = ex2.approx.ftz((s - 1) log2(e) / tau), which flushes results below 2^-126 to zero, and the
# backward scales each row by g exp(1/tau - lse) / tau <= g / (tau E_min) in fp32. For bf16-rounded unit rows
# s >= -(1 + 2^-8)^2, so no term of a row underflows while 2 (1 + 2^-8)^2 log2(e) / tau <= 126 (1/tau <= 43.3), and
# the row scale stays finite for 1/tau <= 40 (exp(2 (1 + 2^-8)^2 40) 40 < 2^128).
MAX_INV_TAU = 40.0


def _check_tau(tau: float) -> float:
    """The fused sweeps evaluate exp(s/tau - 1/tau) with the fixed maximum 1/tau (rows are unit norm) instead of a
    running row maximum; beyond MAX_INV_TAU a row whose similarities are all negative enough (one anchor anti-correlated
    with the batch) would underflow to a zero row sum, where the reference's log_softmax stays finite. Refuse such
    temperatures instead of returning inf."""
    inv_tau = float(1.0 / tau)
    if not 0.0 < inv_tau <= MAX_INV_TAU:
        raise ValueError(f"tau={tau}: the fused contrastive kernels support 1/tau in (0, {MAX_INV_TAU:g}] "
                         f"(the reference's scripts use tau 0.1 and tau2 4.0)")
    return inv_tau


def _links_to_index(train_links, device):
    """train_links is a numpy int32 [B, 2] array in the reference's data loader (src/data.py:41-44) or a tensor."""
    if isinstance(train_links, torch.Tensor):
        links = train_links.to(device=device, dtype=torch.int64)
    else:
        links = torch.from_numpy(np.ascontiguousarray(np.asarray(train_links), dtype=np.int64)).to(device)
    if links.dim() != 2 or links.shape[1] != 2:
        raise ValueError(f"train_links must be [B, 2], got {tuple(links.shape)}")
    return links[:, 0].contiguous(), links[:, 1].contiguous()


class AnchorShard:
    """How the anchors (rows) of an in-batch contrastive loss are split over the ranks of a process group
    (SURVEY 8(e): every rank holds the whole batch of embeddings — the encoder is replicated — and owns a contiguous
    block of `per` anchors of each side, which it sweeps against all 2B columns).

    Exchange steps: forward, one all-gather of the per-anchor (lse, nll) of both sides ([4, per] fp32 per rank);
    backward, with grads="gather", one all-gather of the owned rows of dA and dB ([2, per, D] fp32 per rank) so that
    every rank returns the full, identical gradient (replicas stay in sync without a gradient all-reduce). With
    grads="local" each rank returns only its own rows (zeros elsewhere): the SUM over ranks is the full gradient.
    `be` is the kernel backend (snag_b200.ops; the tests substitute a CPU stand-in to run the host logic under gloo)."""

    def __init__(self, group=None, grads: str = "gather", be=None, world: int | None = None, rank: int | None = None):
        if grads not in ("gather", "local"):
            raise ValueError("grads must be 'gather' or 'local'")
        self.group, self.grads, self.be = group, grads, (ops if be is None else be)
        if group is not None:
            import torch.distributed as dist
            world, rank = dist.get_world_size(group), dist.get_rank(group)
        self.world, self.rank = (1 if world is None else int(world)), (0 if rank is None else int(rank))

    def bounds(self, B: int) -> tuple[int, int, int]:
        """(r0, r1, per): this rank owns anchors [r0, r1); `per` = ceil(B / world) rounded up to 128 (one row block)."""
        per = ops.round_up((B + self.world - 1) // self.world, 128)
        r0 = min(self.rank * per, B)
        return r0, min(r0 + per, B), per

    def all_reduce(self, t: torch.Tensor) -> torch.Tensor:
        """elementwise sum over the ranks (in place)"""
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, group=self.group)
        return t

    def all_gather(self, t: torch.Tensor) -> torch.Tensor:
        """[...] per rank -> [world, ...]"""
        if self.world == 1:
            return t.unsqueeze(0)
        import torch.distributed as dist
        flat = torch.empty((self.world * t.numel(),), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(flat, t.contiguous().reshape(-1), group=self.group)
        return flat.view(self.world, *t.shape)


_UNSHARDED = None


def _unsharded() -> AnchorShard:
    global _UNSHARDED
    if _UNSHARDED is None:
        _UNSHARDED = AnchorShard()
    return _UNSHARDED


# Contraction widths up to ops.FUSED_BWD_MAX_DPAD (the per-modality calls, D = 300) take the fused backward: logits tile
# recomputed, dL/dlogits formed in registers and kept in tensor memory as the A operand of a second tcgen05.mma — no
# [B, 2B] matrix in HBM. Wider tables (the joint embeddings) keep the two-kernel form, where the MMAs dominate anyway.
FUSED_BACKWARD = os.environ.get("SNAG_FUSED_BACKWARD", "1") != "0"      # A/B switch for measurements
# Forward on half the Gram matrix of the stacked rows, all tables of a step in one launch per contraction width
# (ops.icl_fwd_sym); off: two per-side sweeps per table (sim_kernel<EpiIclFwd>), which execute the whole matrix.
SYM_FORWARD = os.environ.get("SNAG_SYM_FORWARD", "1") != "0"
# Tables too wide for the fused backward (the joint embeddings): the forward keeps E = exp(s/tau - 1/tau) of the half
# matrix in bf16 ([2Bp, 2Bp]: 2 GB per table at B = 16 384) and the backward forms dL/dlogits from it with a bandwidth
# kernel instead of a second pass over the 1200- / 1800-wide contraction. Single rank only (off: recompute).
SAVE_E = os.environ.get("SNAG_SAVE_E", "1") != "0"

# What icl_loss contracts (read at every call; icl_loss.forward_many(precision=) and SnagLossLayer(precision=) override
# it per call / per layer): "bf16" rounds the normalised rows to bf16 before every contraction (losses within ~5e-3
# relative of the reference's fp32 arithmetic, gradients within ~2e-2); "fp32" contracts a three-term bf16 split of the
# unrounded rows (snag_b200.loss_fp32: 3x the contraction width, two-kernel backward at every width). ial_loss stays bf16
# (SNAG never calls it).
TRAIN_PRECISION = "bf16"
PRECISIONS = ("bf16", "fp32")


def _check_precision(precision: str) -> str:
    if precision not in PRECISIONS:
        raise ValueError(f"precision={precision!r}: expected one of {PRECISIONS}")
    return precision


class _IclMany(torch.autograd.Function):
    """(idx_l, idx_r [B], emb_0 .. emb_{n-1} [N, D_p] fp32) -> NLL [n, 2, B] (nll_a, nll_b per table): per-row NLL of both
    directions of the in-batch contrastive loss of the L2-normalised rows emb_p[idx_l], emb_p[idx_r], for n embedding
    tables that share one batch of links (the 2 + 2M icl_loss calls of a step, model/SNAG.py:106,147-159), fused on
    the tensor cores; with an AnchorShard of more than one rank every rank sweeps only its own anchors. Gather +
    F.normalize + bf16 cast are one kernel forward (prep_bf16) and one backward (normalize_bwd_scatter), so autograd
    sees a single node from the tables to the NLL vectors; the backward of all narrow tables is ONE launch."""

    @staticmethod
    def forward(ctx, idx_l, idx_r, inv_tau, shard, normalize, *embs):
        be = shard.be
        B = idx_l.numel()
        Bp = ops.round_up(B, 256)
        r0, r1, per = shard.bounds(B)
        saved, outs, dims = [], [], []
        embs = [emb.contiguous() for emb in embs]
        # stacked operands [a ; b ; a], every part zero padded to Bp rows: side a sweeps [b ; a], side b sweeps [a ; b]
        if hasattr(be, "icl_stack_prep"):
            stacks = be.icl_stack_prep(embs, idx_l, idx_r, Bp, normalize)          # all tables in one launch
        else:
            stacks = []
            for emb in embs:
                S3 = torch.zeros((3 * Bp, ops.round_up(emb.shape[1], 64)), dtype=torch.bfloat16, device=emb.device)
                be.prep_bf16(emb, idx_l, normalize=normalize, out=S3[0:Bp])
                be.prep_bf16(emb, idx_r, normalize=normalize, out=S3[Bp:2 * Bp])
                S3[2 * Bp:2 * Bp + B].copy_(S3[0:B])
                stacks.append(S3)
        loc_all = None
        stats = None
        esaved = {}                                       # table -> saved E (wide tables of an unsharded training step)
        if SYM_FORWARD and hasattr(be, "icl_fwd_sym"):
            # sharded: every rank takes a contiguous share of the launch's work units (tiles of the half matrix, not
            # anchors) and one all-reduce of the partial row sums replaces the all-gather of per-anchor results
            stats = [None] * len(embs)
            if SAVE_E and shard.world == 1 and hasattr(be, "icl_g_from_e"):
                for p, S3 in enumerate(stacks):
                    if S3.shape[1] > ops.FUSED_BWD_MAX_DPAD and ctx.needs_input_grad[5 + p]:
                        esaved[p] = torch.empty((2 * Bp, 2 * Bp), dtype=torch.bfloat16, device=S3.device)
            by_width = {}
            for p, S3 in enumerate(stacks):
                by_width.setdefault(S3.shape[1], []).append(p)
            for group in by_width.values():
                for i in range(0, len(group), ops.ICL_SYM_MAX_PROBLEMS):
                    chunk = group[i:i + ops.ICL_SYM_MAX_PROBLEMS]
                    kw = {"esave": [esaved.get(p) for p in chunk]} if esaved else {}
                    res = be.icl_fwd_sym([stacks[p] for p in chunk], B, Bp, inv_tau, shard.rank, shard.world, shard.all_reduce,
                                         **kw)
                    for q, p in enumerate(chunk):
                        stats[p] = res[q]
        elif shard.world > 1:
            # this rank's anchors of every table, then ONE all-gather of the per-anchor (lse, nll) of both sides
            loc_all = torch.zeros((len(embs), 4, per), dtype=torch.float32, device=embs[0].device)
            if r1 > r0:
                nx = r1 - r0
                for p, S3 in enumerate(stacks):
                    la, na, _ = be.icl_side(S3[r0:r0 + nx], S3[Bp:3 * Bp], B, Bp, inv_tau, r0, nx)
                    lb, nb, _ = be.icl_side(S3[Bp + r0:Bp + r0 + nx], S3[0:2 * Bp], B, Bp, inv_tau, r0, nx)
                    loc_all[p, 0, :nx], loc_all[p, 1, :nx], loc_all[p, 2, :nx], loc_all[p, 3, :nx] = la, na, lb, nb
            allv = shard.all_gather(loc_all).permute(1, 2, 0, 3).reshape(len(embs), 4, -1)[:, :, :B].contiguous()   # anchor order
        n = len(embs)
        if stats is not None:
            groups = list(by_width.values())
            if len(groups) == 1 and len(groups[0]) <= ops.ICL_SYM_MAX_PROBLEMS:
                allstats = res                                      # [n, 4, B] of the single launch, already in table order
            else:
                allstats = torch.stack(stats, 0)
        else:
            rows = []
            for p, S3 in enumerate(stacks):
                if shard.world == 1:
                    lse_a, nll_a, _ = be.icl_side(S3[0:Bp], S3[Bp:3 * Bp], B, Bp, inv_tau)
                    lse_b, nll_b, _ = be.icl_side(S3[Bp:2 * Bp], S3[0:2 * Bp], B, Bp, inv_tau)
                    rows.append(torch.stack([lse_a, nll_a, lse_b, nll_b], 0))
                else:
                    rows.append(allv[p])
            allstats = torch.stack(rows, 0)
        lse = allstats[:, 0::2].contiguous()                         # [n, 2, B]
        nll = allstats[:, 1::2].contiguous()
        ctx.save_for_backward(idx_l, idx_r, lse, *stacks, *embs, *[esaved[p] for p in sorted(esaved)], *([nll] if esaved else []))
        ctx.esaved = tuple(sorted(esaved))
        ctx.dims = (B, Bp, inv_tau, bool(normalize), tuple(int(e.shape[1]) for e in embs))
        ctx.shard = shard
        return nll

    @staticmethod
    def backward(ctx, grad):
        idx_l, idx_r, lse, *saved = ctx.saved_tensors
        B, Bp, inv_tau, nrm, dims = ctx.dims
        shard = ctx.shard
        be = shard.be
        n = len(dims)
        stacks, embs = saved[:n], saved[n:2 * n]
        esaved = dict(zip(ctx.esaved, saved[2 * n:]))
        r0, r1, per = shard.bounds(B)
        # row coefficients of every table at once: cr_x = g_x exp(1/tau - lse_x), dg = g_a + g_b   ([n, B] each)
        grad = grad.contiguous().float()
        cr = grad * torch.exp(inv_tau - lse)
        dg_all = grad[:, 0] + grad[:, 1]
        diag_all = None
        if esaved:
            # the cross diagonal of dL/dlogits, g (P_ii - 1) / tau, from the forward's fp32 NLL (P_ii = exp(-nll_i))
            nll_saved = saved[2 * n + len(esaved)]
            diag_all = (grad[:, 0] * torch.expm1(-nll_saved[:, 0]) + grad[:, 1] * torch.expm1(-nll_saved[:, 1])) * inv_tau
            if B % 4:
                diag_all = torch.nn.functional.pad(diag_all, (0, 4 - B % 4))
        if B % 4:                                         # per-table rows must stay 16-byte aligned
            cr = torch.nn.functional.pad(cr, (0, 4 - B % 4))
            dg_all = torch.nn.functional.pad(dg_all, (0, 4 - B % 4))
        probs = []
        for p in range(n):
            if not ctx.needs_input_grad[5 + p]:
                probs.append(None)
                continue
            probs.append(dict(S3=stacks[p], emb=embs[p], D=dims[p], cra=cr[p, 0], crb=cr[p, 1], dg=dg_all[p]))
        # the anchors this rank differentiates: all of them, or its shard (whole blocks of 128 rows inside [0, Bp))
        a0, nx = (0, Bp) if shard.world == 1 else (r0, max(0, min(per, Bp - r0)) if r1 > r0 else 0)
        dz = [None] * n                                   # per problem: (dz_a, dz_b), rows = anchors a0 .. a0 + nx
        if nx > 0:
            fused = [p for p in range(n) if probs[p] is not None and FUSED_BACKWARD and hasattr(be, "icl_bwd_fused")
                     and probs[p]["S3"].shape[1] <= ops.FUSED_BWD_MAX_DPAD]
            by_width = {}
            for p in fused:
                by_width.setdefault(probs[p]["S3"].shape[1], []).append(p)
            for group in by_width.values():
                for i in range(0, len(group), ops.FUSED_BWD_MAX_PROBLEMS):
                    chunk = group[i:i + ops.FUSED_BWD_MAX_PROBLEMS]
                    res = be.icl_bwd_fused([probs[p]["S3"] for p in chunk], [probs[p]["cra"] for p in chunk],
                                           [probs[p]["crb"] for p in chunk], [probs[p]["dg"] for p in chunk], B, Bp, inv_tau,
                                           a0, nx)
                    for p, pair in zip(chunk, res):
                        dz[p] = pair
            for p in range(n):
                if probs[p] is None or dz[p] is not None:
                    continue
                q = probs[p]
                S3, D = q["S3"], q["D"]
                Ya, Yb = S3[Bp:3 * Bp], S3[0:2 * Bp]
                if p in esaved:                               # dL/dlogits from the E the forward kept: no second pass over D
                    Ga = be.icl_g_from_e(esaved[p], 0, B, Bp, q["cra"], q["crb"], diag_all[p], inv_tau)
                    Gb = be.icl_g_from_e(esaved[p], 1, B, Bp, q["crb"], q["cra"], diag_all[p], inv_tau)
                else:
                    Ga = be.icl_bwd_logits(S3[a0:a0 + nx], Ya, B, Bp, inv_tau, q["cra"], q["crb"], q["dg"], a0, nx)   # [nx, 2Bp] bf16
                    Gb = be.icl_bwd_logits(S3[Bp + a0:Bp + a0 + nx], Yb, B, Bp, inv_tau, q["crb"], q["cra"], q["dg"], a0, nx)
                # row i of G carries every term of dL/d(anchor i) — its own softmax row and its appearances as a column
                # in the other rows' softmaxes (the cc / cr_j terms of EpiIclBwd) — so the owned rows of dA, dB are complete
                kp = {"keep_parts": True} if (shard.world == 1 and hasattr(be, "normalize_bwd_scatter_many")) else {}
                if hasattr(be, "grad_contract_rows"):         # the stacked rows as they lie in memory, read MN-major
                    dz[p] = (be.grad_contract_rows(Ga, Ya, nx, D, **kp), be.grad_contract_rows(Gb, Yb, nx, D, **kp))
                else:
                    dz[p] = (be.grad_contract(Ga, Ya.t().contiguous(), nx, D, **kp),
                             be.grad_contract(Gb, Yb.t().contiguous(), nx, D, **kp))
        out = []
        many = hasattr(be, "normalize_bwd_scatter_many")
        live = [p for p in range(n) if probs[p] is not None]
        # one zero-filled allocation for all gradients (each table's block starts 16-byte aligned)
        offs, total_el = {}, 0
        for p in live:
            offs[p] = total_el
            total_el += ops.round_up(probs[p]["emb"].numel(), 4)
        flat_g = torch.zeros((max(total_el, 1),), dtype=torch.float32, device=idx_l.device)
        dembs = {p: flat_g[offs[p]:offs[p] + probs[p]["emb"].numel()].view_as(probs[p]["emb"]) for p in live}

        def scatter(il, ir, pairs):
            """d emb[p] += backward of normalise + gather applied to (dz_a, dz_b) of every live table"""
            if many:                                      # both sides of every table: one launch
                be.normalize_bwd_scatter_many([probs[p]["emb"] for p in live], il, ir, pairs, [dembs[p] for p in live], nrm)
            else:
                for p, (ga, gb) in zip(live, pairs):
                    be.normalize_bwd_scatter(probs[p]["emb"], il, ga, dembs[p], nrm)
                    be.normalize_bwd_scatter(probs[p]["emb"], ir, gb, dembs[p], nrm)

        if live and shard.world == 1:
            if many:
                scatter(idx_l, idx_r, [dz[p] for p in live])
            else:
                scatter(idx_l, idx_r, [tuple(t.sum(0) if t.dim() == 3 else t for t in dz[p]) for p in live])
        elif live:
            # the owned rows of dA, dB of every table in one flat buffer: one all-gather (grads="gather") instead of one
            # per table, then one scatter launch
            sizes = [2 * per * dims[p] for p in live]
            flat = torch.zeros((sum(sizes),), dtype=torch.float32, device=idx_l.device)
            locs, off = [], 0
            for p, sz in zip(live, sizes):
                loc = flat[off:off + sz].view(2, per, dims[p])
                off += sz
                if nx > 0:
                    for s_ in range(2):
                        t = dz[p][s_]
                        loc[s_, :nx] = (t.sum(0) if t.dim() == 3 else t)[:, :dims[p]]
                locs.append(loc)
            if shard.grads == "gather":
                allf = shard.all_gather(flat)                                            # [world, total]
                pairs, off = [], 0
                for p, sz in zip(live, sizes):
                    g = allf[:, off:off + sz].reshape(shard.world, 2, per, dims[p]).permute(1, 0, 2, 3) \
                        .reshape(2, shard.world * per, dims[p])                          # anchor order, contiguous copy
                    off += sz
                    pairs.append((g[0], g[1]))
                scatter(idx_l, idx_r, pairs)
            elif r1 > r0:                 # "local": only the owned anchors' rows; the SUM over ranks is the gradient
                cnt = r1 - r0
                scatter(idx_l[r0:r1].contiguous(), idx_r[r0:r1].contiguous(), [(loc[0, :cnt], loc[1, :cnt]) for loc in locs])
        for p in range(n):
            out.append(dembs.get(p))
        return (None, None, None, None, None, *out)


class _IclPair:
    """One table: (emb, idx_l, idx_r, inv_tau, shard[, normalize]) -> (nll_a, nll_b)."""

    @staticmethod
    def apply(emb, idx_l, idx_r, inv_tau, shard, normalize=True):
        out = _IclMany.apply(idx_l, idx_r, inv_tau, shard, normalize, emb)
        return out[0, 0], out[0, 1]


class icl_loss(nn.Module):
    """model/SNAG_loss.py:31-128."""

    def __init__(self, tau=0.05, ab_weight=0.5, n_view=2, intra_weight=1.0, inversion=False, neg_cross_kg=False):
        super().__init__()
        self.tau = tau
        self.sim = cosine_sim
        self.weight = ab_weight
        self.n_view = n_view
        self.intra_weight = intra_weight
        self.inversion = inversion
        self.neg_cross_kg = neg_cross_kg
        self.shard = None            # AnchorShard, see distribute()
        self.fp32_be = None          # kernel backend of the fp32 route (None: snag_b200.loss_fp32; tests: a CPU stand-in)
        self._fp32_shard = None      # (shard it was made from, the same shard with the fp32 backend)

    def distribute(self, group, grads: str = "gather", be=None):
        """Shard the anchors of every following forward over the ranks of `group` (SURVEY 8(e); BASELINE configs[4]).
        Every rank must call forward with the same batch; the returned loss is identical on all ranks."""
        self.shard = None if group is None else AnchorShard(group, grads, be)
        self._fp32_shard = None
        return self

    def _shard_for(self, precision: str) -> AnchorShard:
        """The anchor shard of this loss with the kernel backend of `precision`."""
        base = self.shard or _unsharded()
        if precision == "bf16":
            return base
        from . import loss_fp32
        be = loss_fp32 if self.fp32_be is None else self.fp32_be
        if self._fp32_shard is None or self._fp32_shard[0] is not base or self._fp32_shard[1].be is not be:
            sh = copy.copy(base)                  # same group, ranks and exchanges; only the kernels differ
            sh.be = be
            self._fp32_shard = (base, sh)
        return self._fp32_shard[1]

    def forward(self, emb, train_links, neg_l=None, neg_r=None, weight_norm=None, norm=True):
        if neg_l is not None or neg_r is not None:
            raise NotImplementedError("explicit negatives (MEAformer replay, MEAformer.py:126) are outside the SNAG path")
        if self.inversion:
            raise NotImplementedError("inversion=True is unreachable from SNAG (model/SNAG.py:50-51)")
        if self.n_view != 2:
            # the reference itself fails here: labels are [B, B*n_view] against logits [B, 2B] (model/SNAG_loss.py:84-89)
            raise RuntimeError(f"n_view={self.n_view}: labels [B, B*n_view] do not match the [B, 2B] logits "
                               f"(model/SNAG_loss.py:84-89 raises as well)")
        return self.forward_many([emb], train_links, [weight_norm], norm=norm)[0]

    def forward_many(self, embs, train_links, weight_norms=None, norm=True, precision=None):
        """The same loss for several embedding tables that share the batch `train_links` (what one SNAG step does 2 + 2M
        times, model/SNAG.py:106,147-159): returns one scalar per table, each equal to forward(emb, train_links,
        weight_norm=w). One autograd node covers all tables, so their backward sweeps are batched into one launch.
        precision: "bf16" or "fp32" (None: TRAIN_PRECISION at the time of the call)."""
        precision = _check_precision(TRAIN_PRECISION if precision is None else precision)
        if self.inversion:
            raise NotImplementedError("inversion=True is unreachable from SNAG (model/SNAG.py:50-51)")
        if self.n_view != 2:
            raise RuntimeError(f"n_view={self.n_view}: labels [B, B*n_view] do not match the [B, 2B] logits "
                               f"(model/SNAG_loss.py:84-89 raises as well)")
        weight_norms = [None] * len(embs) if weight_norms is None else list(weight_norms)
        idx_l, idx_r = _links_to_index(train_links, embs[0].device)
        embs = [e.float() for e in embs]
        inv_tau = _check_tau(self.tau)
        if not norm:
            # model/SNAG_loss.py:59 skips F.normalize (no caller in the reference does: model/SNAG.py:106,147-159; MCLEA.py;
            # MEAformer.py). The sweeps evaluate exp(s/tau - 1/tau) with the fixed maximum 1/tau, i.e. they need |s| <= 1:
            # scale the rows by a power of two 2^-e (exact in fp32 and bf16) so that the largest gathered row has norm <= 1
            # and fold 4^e into the temperature — s/tau is unchanged, term by term.
            with torch.no_grad():
                m2 = max(float(torch.maximum(e.index_select(0, idx_l).square().sum(1).max(),
                                             e.index_select(0, idx_r).square().sum(1).max())) for e in embs)
            e2 = max(0, int(np.ceil(0.5 * np.log2(max(m2, 1e-30)))))
            inv_tau = inv_tau * 4.0 ** e2
            if inv_tau > MAX_INV_TAU:
                raise ValueError(f"norm=False with squared row norms up to {m2:.3g} at tau={self.tau}: logits reach "
                                 f"{inv_tau:.3g}, beyond the fused kernels' range of {MAX_INV_TAU:g}")
            embs = [e * (2.0 ** -e2) for e in embs]
        # normalising only the 2B gathered rows equals normalising all N first (model/SNAG_loss.py:60-64), row by row
        nll = _IclMany.apply(idx_l, idx_r, inv_tau, self._shard_for(precision), bool(norm), *embs)
        batch = idx_l.numel()
        alpha = self.weight
        # softXEnt (:42-54) and the alpha mix (:126) for all tables at once — the same elementwise operations and one
        # reduction per table and side as the reference's per-call code, without 2 + 2M rounds of tiny launches
        weighted = [p for p, w in enumerate(weight_norms) if w is not None]
        if weighted:
            # :66-69 — min over (w[left], w[right]); torch.min along a stacked dim routes the gradient to the first
            # minimum exactly like the reference's torch.min(torch.stack([...], dim=1), 1)[0]
            wn = torch.stack([weight_norms[p] for p in weighted], 0)                                   # [n_w, N]
            wmin = torch.min(torch.stack([wn.index_select(1, idx_l), wn.index_select(1, idx_r)], dim=2), 2)[0]   # [n_w, B]
            if len(weighted) == len(weight_norms):
                w_all = wmin
            else:
                ones = torch.ones((batch,), dtype=wmin.dtype, device=wmin.device)
                it = iter(range(len(weighted)))
                w_all = torch.stack([wmin[next(it)] if w is not None else ones for w in weight_norms], 0)
            per_side = (nll * w_all[:, None, :]).sum(2) / batch                                        # softXEnt :51
        else:
            per_side = nll.sum(2) / batch                                                              # softXEnt :53
        loss = alpha * per_side[:, 0] + (1 - alpha) * per_side[:, 1]                                   # :126
        return list(loss.unbind(0))


class _Contract(torch.autograd.Function):
    """S = P . Q^T (fp32 [n1, D] x [n2, D] -> fp32 [n1, n2]) with operands rounded to bf16, on the tcgen05 mainloop,
    differentiable: dP = dS . Q, dQ = dS^T . P run on the same mainloop."""

    @staticmethod
    def forward(ctx, P, Q):
        Pb, _ = ops.prep_bf16(P.contiguous().float(), None, normalize=False)
        Qb, _ = ops.prep_bf16(Q.contiguous().float(), None, normalize=False)
        ctx.save_for_backward(Pb, Qb)
        ctx.dims = (P.shape[0], Q.shape[0], P.shape[1])
        return ops.contract(Pb, Qb, P.shape[0], Q.shape[0])

    @staticmethod
    def backward(ctx, dS):
        Pb, Qb = ctx.saved_tensors
        n1, n2, D = ctx.dims
        dP = dQ = None
        dSb, _ = ops.prep_bf16(dS.contiguous().float(), None, normalize=False)            # [n1, n2pad]
        if ctx.needs_input_grad[0]:
            Qt = torch.zeros((Qb.shape[1], dSb.shape[1]), dtype=torch.bfloat16, device=dS.device)
            Qt[:, :n2] = Qb[:n2].t()
            dP = ops.contract(dSb, Qt, n1, D)
        if ctx.needs_input_grad[1]:
            dSt, _ = ops.prep_bf16(dS.t().contiguous().float(), None, normalize=False)    # [n2, n1pad]
            Pt = torch.zeros((Pb.shape[1], dSt.shape[1]), dtype=torch.bfloat16, device=dS.device)
            Pt[:, :n1] = Pb[:n1].t()
            dQ = ops.contract(dSt, Pt, n2, D)
        return dP, dQ


class _IalPair(torch.autograd.Function):
    """Row-wise KL( softmax(q_i) || softmax(p_i) ) of both directions for unit rows: p from `src`, q from `tar`
    (detached), logits laid out as in icl_loss ([cross | self with the diagonal masked] / tau).
        KL_i = sum_j Q_ij (q_ij - p_ij) - lse_q_i + lse_p_i ,
        sum_j Q_ij q_ij = (z^t_i . (Q Y^t)_i) / tau ,   sum_j Q_ij p_ij = (z^s_i . (Q Y^s)_i) / tau
    so the forward needs the row log-sum-exps (EpiIclFwd sweeps), Q once in bf16 (EpiIclBwd with row coefficients
    exp(1/tau - lse_q)) and two split-K products with the stacked embeddings. Backward: dL/dp = g (P - Q); both
    probability matrices come from the dL/dlogits sweep with the ICL coefficient pattern (row term + transposed-role
    term, see EpiIclBwd) run once on the src operands and once on the tar operands; their difference is contracted
    with the stacked src embeddings and pushed through the normalise/gather backward."""

    be = ops          # kernel backend (the CPU tests substitute tests/oracle_backend.py to check the host algebra)

    @staticmethod
    def forward(ctx, src, tar, idx_l, idx_r, inv_tau):
        be = _IalPair.be
        src, tar = src.contiguous(), tar.contiguous()
        B = idx_l.numel()
        Bp = ops.round_up(B, 256)
        dev = src.device

        def stack(emb):
            S3 = torch.zeros((3 * Bp, ops.round_up(emb.shape[1], 64)), dtype=torch.bfloat16, device=dev)
            be.prep_bf16(emb, idx_l, normalize=True, out=S3[0:Bp])
            be.prep_bf16(emb, idx_r, normalize=True, out=S3[Bp:2 * Bp])
            S3[2 * Bp:2 * Bp + B].copy_(S3[0:B])
            return S3

        Ss, St = stack(src), stack(tar)
        Ds, Dt = src.shape[1], tar.shape[1]
        zero = torch.zeros((B,), dtype=torch.float32, device=dev)
        sides = ((slice(0, Bp), slice(Bp, 3 * Bp)), (slice(Bp, 2 * Bp), slice(0, 2 * Bp)))     # (anchors, [other ; this])
        lse_p, lse_q, kl = [], [], []
        for xs, ys in sides:
            lp, _, _ = be.icl_side(Ss[xs], Ss[ys], B, Bp, inv_tau)
            lq, _, _ = be.icl_side(St[xs], St[ys], B, Bp, inv_tau)
            crq = (torch.exp(inv_tau - lq) / inv_tau).contiguous()            # EpiIclBwd multiplies by 1/tau: Q = cr E / tau
            Q = be.icl_bwd_logits(St[xs], St[ys], B, Bp, inv_tau, crq, zero, zero, self_cols=False)   # row softmax of q
            if hasattr(be, "grad_contract_rows"):                               # stacked rows read MN-major: no transposed copy
                Ut = be.grad_contract_rows(Q, St[ys], B, Dt)                    # (Q Y^t) [B, Dt]
                Us = be.grad_contract_rows(Q, Ss[ys], B, Ds)
            else:
                Ut = be.grad_contract(Q, St[ys].t().contiguous(), B, Dt)
                Us = be.grad_contract(Q, Ss[ys].t().contiguous(), B, Ds)
            zq = (St[xs][:B, :Dt].float() * Ut).sum(1) * inv_tau
            zp = (Ss[xs][:B, :Ds].float() * Us).sum(1) * inv_tau
            kl.append(zq - zp - lq + lp)
            lse_p.append(lp)
            lse_q.append(lq)
        ctx.save_for_backward(Ss, St, src, idx_l, idx_r, *lse_p, *lse_q)
        ctx.dims = (B, Bp, Ds, inv_tau)
        return kl[0], kl[1]

    @staticmethod
    def backward(ctx, g_a, g_b):
        Ss, St, src, idx_l, idx_r, lpa, lpb, lqa, lqb = ctx.saved_tensors
        B, Bp, Ds, inv_tau = ctx.dims
        be = _IalPair.be
        dev = Ss.device
        g_a = torch.zeros_like(lpa) if g_a is None else g_a.contiguous().float()
        g_b = torch.zeros_like(lpb) if g_b is None else g_b.contiguous().float()
        zero = torch.zeros((B,), dtype=torch.float32, device=dev)
        cpa, cpb = (g_a * torch.exp(inv_tau - lpa)).contiguous(), (g_b * torch.exp(inv_tau - lpb)).contiguous()
        cqa, cqb = (g_a * torch.exp(inv_tau - lqa)).contiguous(), (g_b * torch.exp(inv_tau - lqb)).contiguous()
        demb = torch.zeros_like(src)
        # Both matrices are written centred on E(s = 0) = exp(-1/tau): at tau = 4 the softmaxes are within a few per cent
        # of uniform, and rounding P and Q to bf16 before subtracting them would leave ~20 % noise on P - Q. The part
        # removed by the centring, ebar/tau * (dr_i + dc_j) over the unmasked columns, is rank one and is added back to
        # G . Y in fp32 below.
        ebar = float(np.exp(-inv_tau))
        sides = ((slice(0, Bp), slice(Bp, 3 * Bp), cpa, cpb, cqa, cqb, idx_l),
                 (slice(Bp, 2 * Bp), slice(0, 2 * Bp), cpb, cpa, cqb, cqa, idx_r))
        for xs, ys, cp_row, cp_col, cq_row, cq_col, idx in sides:
            Gs = be.icl_bwd_logits(Ss[xs], Ss[ys], B, Bp, inv_tau, cp_row, cp_col, zero, ebar=ebar)   # g (P + transposed-role P) / tau
            Gt = be.icl_bwd_logits(St[xs], St[ys], B, Bp, inv_tau, cq_row, cq_col, zero, ebar=ebar)   # the same for Q
            dz = be.grad_contract_rows(Gs - Gt, Ss[ys], B, Ds) if hasattr(be, "grad_contract_rows") else \
                be.grad_contract(Gs - Gt, Ss[ys].t().contiguous(), B, Ds)
            Y0 = Ss[ys][:B, :Ds].float()                       # cross columns: the other side
            Y1 = Ss[ys][Bp:Bp + B, :Ds].float()                # self columns: this side (column i is masked for row i)
            dr, dc0, dc1 = cp_row - cq_row, cp_col - cq_col, cp_row - cq_row
            common = dr[:, None] * (Y0.sum(0) + Y1.sum(0))[None, :] - dr[:, None] * Y1 \
                + (dc0 @ Y0 + dc1 @ Y1)[None, :] - dc1[:, None] * Y1
            dz = dz + (ebar * inv_tau) * common
            be.normalize_bwd_scatter(src, idx, dz.contiguous(), demb, True)
        return demb, None, None, None, None


class ial_loss(nn.Module):
    """model/SNAG_loss.py:130-202 — unimodal/multimodal KL alignment loss."""

    def __init__(self, tau=0.05, ab_weight=0.5, zoom=0.1, n_view=2, inversion=False, reduction="mean", detach=False):
        super().__init__()
        self.tau = tau
        self.sim = cosine_sim
        self.weight = ab_weight
        self.zoom = zoom
        self.n_view = n_view
        self.inversion = inversion
        self.reduction = reduction
        self.detach = detach

    def forward(self, src_emb, tar_emb, train_links, norm=True):
        if self.inversion:
            raise NotImplementedError("inversion=True is unreachable from SNAG / MCLEA")
        if not norm:
            # no caller in the reference passes norm=False (model/MCLEA.py:128-139)
            raise NotImplementedError("norm=False: the fused kernel relies on unit rows (logits bounded by 1/tau)")
        if self.reduction not in ("mean", "sum"):
            # the reference returns zoom * (alpha * [B, 2B] matrix + ...) here (model/SNAG_loss.py:195-202): an unreduced
            # matrix is exactly what the fused path never forms
            raise NotImplementedError(f"reduction={self.reduction!r}: only 'mean' and 'sum' (config.py:103's choices)")
        idx_l, idx_r = _links_to_index(train_links, src_emb.device)
        kl_a, kl_b = _IalPair.apply(src_emb.float(), tar_emb.detach().float(), idx_l, idx_r, _check_tau(self.tau))
        batch = idx_l.numel()
        denom = float(batch * 2 * batch) if self.reduction == "mean" else 1.0     # .mean() runs over the [B, 2B] matrix (:195-197)
        alpha = self.weight
        return self.zoom * (alpha * kl_a.sum() / denom + (1 - alpha) * kl_b.sum() / denom)


class SnagLossLayer(nn.Module):
    """The loss half of SNAG.forward (model/SNAG.py:104-116, 140-160) as one module, with the reference's member names:
    GMI = criterion_cl_joint(joint_emb) + criterion_cl_joint(joint_emb_fz); ECIA = inner_view_loss over the modality
    embeddings with the per-modality weights; IIR = inner_view_loss over the hidden-state embeddings;
    multi_loss_layer (CustomMultiLossLayer, 6) inside inner_view_loss; multi_loss_layer_2 (AutomaticWeightedLoss, 7) on
    top when `awloss` — off by default like --awloss (config.py:114), i.e. the three terms are summed. (With --awloss 1
    the reference passes the LIST as one positional argument, model/SNAG.py:117, which raises a TypeError inside
    AutomaticWeightedLoss.forward; here the three terms are passed as the three arguments its signature expects.)
    That is 2 + 2M icl_loss calls per step for M present modalities — the "loss-layer slice" bench.py times.
    `streams` / `hidden` are 6-tuples ordered (gph, rel, att, img, name, char) with None for absent modalities."""

    WEIGHT_COLUMN = (3, 2, 1, 0, 4, 5)      # model/SNAG.py:145-150: gph<-w[:,3], rel<-w[:,2], att<-w[:,1], img<-w[:,0], ...

    def __init__(self, tau=0.1, ab_weight=0.5, awloss=False, precision=None):
        super().__init__()
        self.awloss = awloss
        # what the icl_loss calls contract ("bf16" / "fp32"; None: loss.TRAIN_PRECISION at the time of each call)
        self.precision = None if precision is None else _check_precision(precision)
        self.multi_loss_layer = CustomMultiLossLayer(loss_num=6)                         # model/SNAG.py:48
        self.multi_loss_layer_2 = AutomaticWeightedLoss(num=7)                           # :49
        self.criterion_cl = icl_loss(tau=tau, ab_weight=ab_weight, n_view=2)             # :50
        self.criterion_cl_joint = icl_loss(tau=tau, ab_weight=ab_weight, n_view=2)       # :51

    def distribute(self, group, grads: str = "gather"):
        self.criterion_cl.distribute(group, grads)
        self.criterion_cl_joint.distribute(group, grads)
        return self

    def inner_view_loss(self, streams, train_ill, weight_norm=None, losses=None):
        """model/SNAG.py:140-160; `losses` = the per-stream icl_loss values when they were already evaluated in a batch."""
        if losses is None:
            present = [(emb, col) for emb, col in zip(streams, self.WEIGHT_COLUMN) if emb is not None]
            wn = None if weight_norm is None else weight_norm * weight_norm.shape[1]
            vals = self.criterion_cl.forward_many([e for e, _ in present], train_ill,
                                                  [None if wn is None else wn[:, c] for _, c in present],
                                                  precision=self.precision)
            it = iter(vals)
            losses = [0 if emb is None else next(it) for emb in streams]
        return self.multi_loss_layer(losses)

    def forward(self, streams, hidden, joint_emb, joint_emb_fz, batch, weight_norm):
        # all 2 + 2M calls of the step share the batch: one autograd node, so that the backward of the narrow tables is a
        # single fused launch (criterion_cl and criterion_cl_joint have the same tau / ab_weight, model/SNAG.py:50-51)
        wn = weight_norm * weight_norm.shape[1]
        s_pres = [(e, c) for e, c in zip(streams, self.WEIGHT_COLUMN) if e is not None]
        h_pres = [h for h in hidden if h is not None]
        vals = self.criterion_cl.forward_many([joint_emb, joint_emb_fz] + [e for e, _ in s_pres] + h_pres, batch,
                                              [None, None] + [wn[:, c] for _, c in s_pres] + [None] * len(h_pres),
                                              precision=self.precision)
        gmi = vals[0] + vals[1]
        it = iter(vals[2:])
        ecia = self.inner_view_loss(streams, batch, losses=[0 if e is None else next(it) for e in streams])
        iir = self.inner_view_loss(hidden, batch, losses=[0 if h is None else next(it) for h in hidden])
        loss_list = [gmi, ecia, iir]
        return self.multi_loss_layer_2(*loss_list) if self.awloss else sum(loss_list)     # :116-119
