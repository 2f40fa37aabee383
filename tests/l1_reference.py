"""Host references of the --distance 1 evaluation for sizes whose [n, n] matrix the host cannot hold: a streaming
evaluation over row blocks and an audit of selected entities, both on oracle.l1_distance (fp64 index-order sums rounded
once) with the same per-element arithmetic as oracle.align_eval_l1. TEST-ONLY."""
from __future__ import annotations

import numpy as np

from oracle import oracle

_ONE, _TWO = np.float32(1.0), np.float32(2.0)


def _mean_desc(top_desc: np.ndarray, k: int) -> np.ndarray:
    """Mean of the k largest, summed largest first in fp32 (src/utils.py:431-432 as the oracle evaluates it)."""
    s = np.zeros(top_desc.shape[:-1], np.float32)
    for t in range(k):
        s = (s + top_desc[..., t]).astype(np.float32)
    return (s / np.float32(k)).astype(np.float32)


def _chain(d: np.ndarray, nv1, nv2) -> np.ndarray:
    """1 - ((2 (1 - d) - nv1) - nv2) in fp32, one rounding per op (main.py:393 then 1 - csls)."""
    c = (_ONE - d).astype(np.float32)
    u = (_TWO * c - nv1).astype(np.float32)
    return (_ONE - (u - nv2).astype(np.float32)).astype(np.float32)


def align_eval_l1_stream(x: np.ndarray, y: np.ndarray, csls: bool = True, k: int = 10, block_rows: int = 1024) -> dict:
    """oracle.align_eval_l1 without the [n, n] matrix (three passes over row blocks; no top-3)."""
    x, y = np.ascontiguousarray(x, np.float32), np.ascontiguousarray(y, np.float32)
    n = x.shape[0]
    if y.shape != x.shape:
        raise ValueError("x and y must have the same shape")
    if csls and k > n:
        raise RuntimeError("selected index k out of range")
    blocks = [(r0, min(n, r0 + block_rows)) for r0 in range(0, n, block_rows)]
    nv1 = nv2 = None
    if csls:
        nv1 = np.empty((n,), np.float32)
        col_top = np.full((k, n), -np.inf, np.float32)
        for r0, r1 in blocks:
            c = (_ONE - oracle.l1_distance(x[r0:r1], y)).astype(np.float32)
            nv1[r0:r1] = _mean_desc(-np.sort(-c, axis=1)[:, :k], k)
            both = np.concatenate([col_top, c], 0)
            col_top = -np.sort(-both, axis=0)[:k]
        nv2 = _mean_desc(col_top.T, k)
    g = np.empty((n,), np.float32)
    for r0, r1 in blocks:
        d = np.diag(oracle.l1_distance(x[r0:r1], y[r0:r1])).astype(np.float32)
        g[r0:r1] = _chain(d, nv1[r0:r1], nv2[r0:r1]) if csls else d
    l2r = np.empty((n,), np.int32)
    r2l = np.zeros((n,), np.int64)
    cols = np.arange(n)
    for r0, r1 in blocks:
        d = oracle.l1_distance(x[r0:r1], y)
        dist = _chain(d, nv1[r0:r1, None], nv2[None, :]) if csls else d
        rows = np.arange(r0, r1)[:, None]
        gr = g[r0:r1, None]
        l2r[r0:r1] = ((dist < gr) | ((dist == gr) & (cols[None, :] < rows))).sum(1)
        gc = g[None, :]
        r2l += ((dist < gc) | ((dist == gc) & (rows < cols[None, :]))).sum(0)
    out = dict(rank_l2r=l2r, rank_r2l=r2l.astype(np.int32), g=g)
    if csls:
        out.update(nv1=nv1, nv2=nv2)
    return out


def audit_l1(xs: np.ndarray, other: np.ndarray, self_id, csls: bool, k: int, nv_other, transposed: bool) -> dict:
    """Selected entities `xs` (pair ids `self_id`) of one side against ALL of the other side: their own neighbourhood
    mean, ground-truth distance and rank, given the other side's neighbourhood means. transposed=False: xs are sources
    (rows of the distance matrix); True: targets (columns)."""
    xs, other = np.ascontiguousarray(xs, np.float32), np.ascontiguousarray(other, np.float32)
    sid = np.asarray(self_id, np.int64)
    d = oracle.l1_distance(xs, other)                        # |x - y| is symmetric: the same values either way round
    nv = np.zeros((xs.shape[0],), np.float32)
    if csls:
        nv = _mean_desc(-np.sort(-(_ONE - d).astype(np.float32), axis=1)[:, :k], k)
        nvo = np.asarray(nv_other, np.float32)[None, :]
        dist = _chain(d, nvo, nv[:, None]) if transposed else _chain(d, nv[:, None], nvo)
    else:
        dist = d
    rows = np.arange(xs.shape[0])
    g = dist[rows, sid]
    others = np.arange(other.shape[0])[None, :]
    rank = ((dist < g[:, None]) | ((dist == g[:, None]) & (others < sid[:, None]))).sum(1).astype(np.int32)
    return dict(nv=nv, g=g, rank=rank)
