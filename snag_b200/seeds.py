"""Unsupervised seed induction — SURVEY 8(f) rank 4: host-side mirror of visual_pivot_induction
(SNAG_MMEA/src/data.py:367-402) and get_topk_indices (SNAG_MMEA/src/utils.py:437-443).

The reference forms the full [n_left, n_right] similarity matrix of the (L2-normalised) image / name / char features,
takes the K = 100 * unsup_k largest entries with torch.topk over the flattened matrix and greedily keeps pairs whose
entities are still unused. Here the matrix is never formed:
  1. one top-k sweep (sim_kernel<EpiRowTopK>) gives every left entity's 16 best scores; the K-th largest of that pool,
     lowered by the tensor-core error bound, is a lower bound of the tensor-core score of every entry whose canonical
     score is among the K largest of the whole matrix (see _admission_threshold);
  2. one thresholded sweep (sim_kernel<EpiRowColTopK> with that bound as every column's admission threshold) streams
     out every entry at or above it — a superset of the global top K;
  3. the collected entries are re-scored with the canonical dot product (fp64, index order), sorted by
     (similarity descending, flat index ascending) and cut to K;
  4. the greedy matching runs on the host exactly as in the reference (sets instead of list scans).
Operands are the bf16-rounded features (precision="bf16", the same contract as the evaluation path) or the unrounded
fp32 features (precision="fp32": split-bf16 sweeps and fp32 canonical re-scores of snag_b200.fp32), as the reference
ranks them.
"""
from __future__ import annotations

import numpy as np
import torch

from . import mining
from . import ops as _cuda_ops
from ._lib import KT, SnagError
from .evaluate import _check_precision


def _admission_threshold(pool_kth: torch.Tensor, eps: float) -> torch.Tensor:
    """Admission threshold (in the sweep's score c = 2 s - 1) of the thresholded sweep, from the K-th largest
    tensor-core score of the pool and eps, the backend's bound of |s_tensor_core - s_canonical| (tc_margin of the real
    operands). The pool holds K entries with c_tc >= pool_kth, so K entries have s_canonical >= (1 + pool_kth)/2 - eps
    and every entry of the canonical top K has at least that s_canonical, hence s_tc >= (1 + pool_kth)/2 - 2 eps:
    c_tc >= pool_kth - 4 eps (a margin eps in s is 2 eps in c). eps includes 1e-6 for the fp32 roundings of c."""
    return pool_kth - 4.0 * eps


def topk_similarity_entries(left_f: torch.Tensor, right_f: torch.Tensor, K: int, _backend=None, precision: str = "bf16"):
    """(rows int64 [K'], cols int64 [K'], sims fp32 [K']) — the K' = min(K, n_l * n_r) largest entries of
    left_f @ right_f.T in descending order, ties by ascending flat index (get_topk_indices, src/utils.py:437-443).
    precision: "bf16" (default) ranks the features rounded to bf16, "fp32" the unrounded fp32 features."""
    _check_precision(precision)
    be = mining._backend_for(precision, _backend)
    n_l, n_r = left_f.shape[0], right_f.shape[0]
    K = min(int(K), n_l * n_r)
    if K <= 0:
        raise ValueError("K must be positive")
    X, xn = mining._prep(be, precision, left_f, False, 0)
    Y, yn = mining._prep(be, precision, right_f, False, 1)
    dev = X.device
    # with unit "norms" the sweep's score c = 1 - clamp(2 - 2 s, 0) = 2 s - 1 is monotone in s (s <= 1)
    one_l = torch.ones((n_l,), dtype=torch.float32, device=dev)
    one_r = torch.ones((n_r,), dtype=torch.float32, device=dev)
    part = be.eval_rowtopk(X, Y, one_l, one_r, n_l, n_r)
    _, pool = be.topk_merge_mean(part, 1, want_nv=False, want_cand=True)               # [n_l, KT]
    pool = pool.reshape(-1)
    pool = pool[torch.isfinite(pool)]
    if pool.numel() < K:
        # more entries requested than the per-row pools hold (K > 16 * n_left): every entry qualifies
        thr = torch.tensor(float("-inf"), device=dev)
    else:
        eps = be.tc_margin(X.shape[1], float(torch.sqrt(xn.max() * yn.max()).item()))
        thr = _admission_threshold(torch.topk(pool, K).values[-1], eps)
    colthr = torch.full((n_r,), float(thr), dtype=torch.float32, device=dev)
    colb = (0.5 * colthr - 4e-6).contiguous()                                       # s > (yn - 1 + thr)/2 with yn = 1
    n_ctas = int(_cuda_ops._lib.load().snag_num_sms()) if _backend is None else 148
    cap = _cuda_ops.round_up(int(2.5 * max(K, 4096) / n_ctas) + 4096, 1024)
    # 12 bytes per stream entry (int64 column + c, int32 row) in n_ctas CTA-private streams, whatever the width
    while True:
        _, _, stream, stream_row, stream_cnt = be.eval_rowcoltopk(X, Y, one_l, one_r, n_l, n_r, colthr, colb, cap)
        cnt = stream_cnt.to(torch.int64)
        if int(cnt.max().item()) <= cap:
            break
        cap *= 4                                                                   # a stream filled up (its counter saturates
                                                                                   # just above the capacity): enlarge and redo
        if cap * stream.shape[0] * 12 > (32 << 30):
            raise SnagError("topk_similarity_entries: too many entries above the threshold (degenerate similarities)")
    keep = torch.arange(stream.shape[1], device=dev)[None, :] < cnt[:, None]
    cols = (stream[keep] & 0xFFFFFFFF).to(torch.int32).contiguous()
    rows = stream_row[keep].contiguous()
    sims = be.pairs_dot(X, Y, rows, cols)
    flat = rows.to(torch.int64) * n_r + cols.to(torch.int64)
    order = torch.argsort(flat)                                                      # ties by ascending flat index:
    order = order[torch.argsort(sims[order], descending=True, stable=True)]          # stable sort on the similarity
    order = order[:K]
    if order.numel() < K:
        raise SnagError("topk_similarity_entries: the thresholded sweep returned fewer than K entries")
    return rows[order].to(torch.int64), cols[order].to(torch.int64), sims[order]


def visual_pivot_induction(args, left_ents, right_ents, img_features, ills, logger):
    """Drop-in for src/data.visual_pivot_induction (same signature, same log lines, same int32 [n, 2] result); ranks in
    mining.LINK_PRECISION."""
    dev = torch.device("cuda", torch.cuda.current_device())
    feats = torch.as_tensor(img_features, dtype=torch.float32)
    l_img_f = feats[torch.as_tensor(list(left_ents), dtype=torch.int64)].to(dev)
    r_img_f = feats[torch.as_tensor(list(right_ents), dtype=torch.int64)].to(dev)
    topk = args.unsup_k
    rows, cols, sims = topk_similarity_entries(l_img_f, r_img_f, topk * 100, precision=mining.LINK_PRECISION)
    print("highest sim:", sims[0].item(), "lowest sim:", sims[-1].item())              # src/utils.py:441
    rows, cols = rows.cpu().tolist(), cols.cpu().tolist()
    visual_links = []
    used = set()
    for r, c in zip(rows, cols):                                                      # src/data.py:381-394
        le, re = left_ents[r], right_ents[c]
        if le in used or re in used:
            continue
        used.add(le)
        used.add(re)
        visual_links.append((le, re))
        if len(visual_links) == topk:
            break
    ill_set = set((int(a), int(b)) for a, b in ills)
    count = float(sum(1 for link in visual_links if (int(link[0]), int(link[1])) in ill_set))
    logger.info(f"{(count / len(visual_links) * 100):.2f}% in true links")
    logger.info(f"visual links length: {(len(visual_links))}")
    return np.array(visual_links, dtype=np.int32)
