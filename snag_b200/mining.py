"""Iterative-learning link mining — host-side mirror of SNAG.Iter_new_links (SNAG_MMEA/model/SNAG.py:192-208,
driver main.py:214-223): mutual nearest neighbours between the non-train entities of the two graphs.

The reference concatenates pairwise_distances over 1000-row slabs into a [n_left, n_right] fp32 matrix, takes
torch.argmin along both axes and filters the pairs with Python list logic (O(n * |links|) membership tests).
Here one fused tcgen05 sweep produces both argmin vectors (the matrix is never formed) and the link filtering is
integer tensor work. Same arithmetic contract as the evaluation: d_ij follows src/utils.py:210-218 op by op in fp32,
ties go to the lowest index like torch.argmin, and the operands are the bf16-rounded rows (precision="bf16") or the
unrounded fp32 rows (precision="fp32", the snag_b200.fp32 backend: split-bf16 sweeps, canonical re-scores on the fp32
rows), as the reference mines them.
"""
from __future__ import annotations

import torch

from . import fp32 as _fp32
from . import ops as _cuda_ops
from ._lib import KT, SnagError
from .evaluate import _check_precision

# What the trainer's link searches run on: Iter_new_links here and seeds.visual_pivot_induction
# (python -m snag_b200.patch --link-precision fp32 sets it).
LINK_PRECISION = "bf16"


def _backend_for(precision: str, _backend=None):
    """The kernel backend of `precision`; _backend is a test seam (tests/oracle_backend.py), the product never passes it."""
    if _backend is not None:
        return _backend
    return _fp32 if precision == "fp32" else _cuda_ops


def _prep(be, precision: str, t: torch.Tensor, normalize: bool, side: int):
    """(operand, ||row||^2) of `t` for the backend of `precision`; side 0 = the sweeps' sources, 1 = their targets (the
    layout of fp32.prep's split operand; bf16 operands have one layout)."""
    if precision == "fp32":
        return be.prep(t.contiguous().float(), None, normalize, side)
    return be.prep_bf16(t.contiguous().float(), None, normalize)


def mutual_nearest(x: torch.Tensor, y: torch.Tensor, normalize: bool = False, _backend=None, canonical: bool = True,
                   precision: str = "bf16"):
    """(preds_l int64 [n1], preds_r int64 [n2], dmin_l fp32 [n1], dmin_r fp32 [n2]): for every row of x its nearest row
    of y under the squared distance of src/utils.pairwise_distances, and vice versa.

    canonical (default): the tensor cores pick each row's / column's 16 nearest candidates (two top-k sweeps, ids
    tracked); the candidates are re-scored with the oracle's arithmetic (fp64 index-order dot, fp32 clamp chain) and
    the argmin — lowest index on ties, like torch.argmin — is taken over them, with the same verification bound and
    exhaustive completion as the CSLS neighbourhoods. The result does not depend on the MMA accumulation order.
    canonical=False: the single fused sweep (sim_kernel<EpiMutualNN>) that takes both argmins straight from the
    tensor-core distances — exact ties still go to the lowest index, near-ties (< 1e-6) follow the tensor core.
    precision: "bf16" (default) mines the rows rounded to bf16; "fp32" mines the unrounded fp32 rows (canonical only):
    argmins and minima are the oracle's on those rows."""
    _check_precision(precision)
    if precision == "fp32" and not canonical:
        raise ValueError("canonical=False (the fused EpiMutualNN sweep) mines bf16 operands only")
    be = _backend_for(precision, _backend)
    n1, n2 = x.shape[0], y.shape[0]
    X, xn = _prep(be, precision, x, normalize, 0)
    Y, yn = _prep(be, precision, y, normalize, 1)      # the split pairing is positional: the swapped sweep works as well
    if canonical and hasattr(be, "topk_rescore"):
        out = []
        for A, B, an, bn, na, nb, tag in ((X, Y, xn, yn, n1, n2, "mine_rows"), (Y, X, yn, xn, n2, n1, "mine_cols")):
            part, pidx = be.eval_rowtopk(A, B, an, bn, na, nb, want_idx=True)
            _, cand, cidx = be.topk_merge_mean(part, 1, want_nv=False, part_idx=pidx)
            _, best_d, best_i = be.topk_rescore(A, B, an, bn, cidx, cand, 1, nb, tag, want_best=True)
            out.append((best_i.to(torch.int64), best_d))
        return out[0][0], out[1][0], out[0][1], out[1][1]
    # upper bound of every column's minimum from a sample of the rows (all of them when there are few): the swapped
    # top-k sweep keeps, per column, the largest c = 1 - d over the sample in registers
    m = n1 if n1 <= 8192 else max(8192, (n1 // 16 + 255) // 256 * 256)
    if m < n1:
        sel = torch.randperm(n1, generator=torch.Generator(device="cpu").manual_seed(3408))[:m].sort()[0].to(x.device)
        Xs, xns = X.index_select(0, sel), xn.index_select(0, sel)
    else:
        Xs, xns = X, xn
    part = be.eval_rowtopk(Y, Xs, yn, xns, n2, m)
    _, cand = be.topk_merge_mean(part, 1, want_nv=False, want_cand=True)
    ub = (1.0 - cand[:, KT - 1]) + 4e-6                       # c = fl(1 - d): d <= 1 - c + rounding
    colb = (0.5 * (yn - ub) - 4e-6).contiguous()
    row_val, row_idx, colkey = be.mutual_nn(X, Y, xn, yn, n1, n2, colb)
    if bool((colkey == -1).any()):
        raise SnagError("mutual_nn: a column received no candidate (pre-filter bound violated)")
    # rows: lexicographic (d, column) minimum over the partial lists
    dmin_l = row_val.min(0)[0]
    big = torch.iinfo(torch.int32).max
    preds_l = torch.where(row_val == dmin_l[None, :], row_idx, torch.full_like(row_idx, big)).min(0)[0].to(torch.int64)
    preds_r = colkey & 0xFFFFFFFF
    dmin_r = (colkey >> 32).to(torch.int32).view(torch.float32)
    return preds_l, preds_r, dmin_l, dmin_r


def iter_new_links(left_non_train, right_non_train, final_emb: torch.Tensor, new_links, refresh: bool, _backend=None,
                   precision: str = "bf16"):
    """Body of Iter_new_links: mutual nearest pairs; when `refresh` is False only those already in `new_links` survive
    (model/SNAG.py:203-206). Entity ids in, list of (left id, right id) tuples out, in increasing order of the position
    in `left_non_train` (the order of the reference's list comprehension). precision: as mutual_nearest."""
    _check_precision(precision)
    if len(left_non_train) == 0 or len(right_non_train) == 0:
        return new_links
    dev = final_emb.device
    left = torch.as_tensor(list(left_non_train), dtype=torch.int64, device=dev)
    right = torch.as_tensor(list(right_non_train), dtype=torch.int64, device=dev)
    preds_l, preds_r, _, _ = mutual_nearest(final_emb.index_select(0, left), final_emb.index_select(0, right),
                                            _backend=_backend, precision=precision)
    pos = torch.arange(left.numel(), device=dev)
    keep = preds_r[preds_l] == pos
    pl, pr = left[keep], right[preds_l[keep]]
    if not refresh:
        n_ent = int(final_emb.shape[0])
        prev = torch.as_tensor([a * n_ent + b for a, b in new_links], dtype=torch.int64, device=dev)
        sel = torch.isin(pl * n_ent + pr, prev)
        pl, pr = pl[sel], pr[sel]
    return list(zip(pl.tolist(), pr.tolist()))


def Iter_new_links(self, epoch, left_non_train, final_emb, right_non_train, new_links=[]):
    """Drop-in for SNAG.Iter_new_links (same signature; installed on the reference class by snag_b200.patch). Mines in
    LINK_PRECISION."""
    step = self.args.semi_learn_step
    return iter_new_links(left_non_train, right_non_train, final_emb, new_links, (epoch + 1) % (step * 5) == step,
                          precision=LINK_PRECISION)
