"""The edge table of the fused evaluation, shared by tests/test_eval_edges_gpu.py (the kernels of every route) and
tests/test_eval_edges_cpu.py (the same driver on the CPU stand-ins), and the comparison with the oracle both use.

The table is a covering design, not a Cartesian product: every n of N_EDGES meets two widths of D_EDGES and every width
meets at least two n, on each route, with a route-dependent shift so that the three routes pair them differently.
CSLS on / off, k and the entry path cycle along the table."""
from __future__ import annotations

import numpy as np

from oracle import oracle
from snag_b200 import evaluate

ROUTES = ("bf16", "fp32", "l1")
# below one 128-row tile, across it, across the 256-wide column tiles and the shard alignment, and above
N_EDGES = (1, 2, 3, 17, 127, 128, 129, 255, 256, 257, 511, 513, 1031)
# across Dpad = 64, the prologue's register-window switch (512), the last width it keeps in registers (2048) and
# beyond; 63 / 64 / 65, 512 / 513 and 2048 / 2049 also cross the L1 operand's multiple of 8
D_EDGES = (1, 3, 8, 63, 64, 65, 97, 512, 513, 2048, 2049, 4096)
PATHS = {"bf16": ("generator", "lazy", "graph"), "fp32": ("generator", "entry"), "l1": ("entry", "generator")}
DEGENERATE = ("zero_rows", "repeated_rows", "one_row", "one_hot")


def edge_cases(route: str, n_max: int | None = None) -> list[tuple]:
    """(n, d, csls, k, want_top3, path) of `route`: 26 cases, each n with two widths."""
    off = 5 * ROUTES.index(route)
    paths = PATHS[route]
    out = []
    for i, n in enumerate(N_EDGES):
        if n_max is not None and n > n_max:
            continue
        for j in range(2):
            t = 2 * i + j
            d = D_EDGES[(t + off) % len(D_EDGES)]
            k = min((1, 3, 16, n if n <= 16 else 10)[t % 4], n)      # k = n for every n <= 3
            out.append((n, d, t % 3 != 2, k, n >= 3, paths[(i + j) % len(paths)]))
    return out


def sharded_cases(route: str) -> list[tuple]:
    """(n, d, world, csls, k): sizes at which a trailing rank owns one target or none (shard_bounds aligns to 256)."""
    off = 3 * ROUTES.index(route)
    sizes = ((17, 3), (129, 2), (257, 8), (513, 3), (255, 2), (1031, 8))
    return [(n, D_EDGES[(2 * q + 1 + off) % len(D_EDGES)], w, q % 3 != 1, (10, 3, 16)[q % 3])
            for q, (n, w) in enumerate(sizes)]


def shard_sizes(n: int, world: int) -> list[int]:
    return [c1 - c0 for c0, c1 in (evaluate.shard_bounds(n, world, r) for r in range(world))]


def degenerate_cases(route: str) -> list[tuple]:
    """(table, n, d): each table at n = 257 and 1031 and at both widths 64 and 97."""
    out = []
    for t, name in enumerate(DEGENERATE):
        for n, d in (((257, 64), (1031, 97)) if t % 2 == 0 else ((257, 97), (1031, 64))):
            out.append((name, n, d))
    return out


def clustered(n: int, d: int, sigma: float, seed: int):
    """Sources around 64 centres and noisy copies of them as targets, normalised as F.normalize does, fp32."""
    rng = np.random.RandomState(seed)
    centres = rng.randn(64, d).astype(np.float32)
    x = rng.randn(n, d).astype(np.float32) + centres[rng.randint(0, 64, n)]
    y = x + np.float32(sigma) * rng.randn(n, d).astype(np.float32)
    return oracle.normalize_rows(x), oracle.normalize_rows(y)


def degenerate(name: str, n: int, d: int, seed: int):
    """The degenerate tables, normalised fp32 rows:
    zero_rows      some sources and targets are all zeros (their distances are the other side's norms);
    repeated_rows  every third source and every fifth target repeats a neighbour: exact ties, the lower index first;
    one_row        both sides are one row repeated: every element ties with its ground truth;
    one_hot        unit basis vectors, half the pairs matched: distances 0 or 2, ties everywhere."""
    rng = np.random.RandomState(seed)
    if name == "one_hot":
        a = rng.randint(0, d, n)
        b = np.where(rng.rand(n) < 0.5, a, rng.randint(0, d, n))
        eye = np.eye(d, dtype=np.float32)
        return eye[a].copy(), eye[b].copy()
    x, y = clustered(n, d, 1.0, seed)
    if name == "zero_rows":
        x[::17] = 0.0
        y[5::23] = 0.0
    elif name == "repeated_rows":
        x[1::3] = x[0::3][:len(x[1::3])]
        y[2::5] = y[1::5][:len(y[2::5])]
        y[3::11] = x[3::11]
    elif name == "one_row":
        x[:] = x[:1]
        y[:] = x[:1]
    else:
        raise ValueError(name)
    return x, y


def top3_checkable(ref: dict, eps: float) -> np.ndarray:
    """Rows whose canonical top 3 the tensor-core routes must reproduce: the 4 nearest candidates by the tensor-core score
    are re-scored canonically, so a row is decided unless its 3rd and 5th nearest lie within the sweep's error of each
    other (eps in s is 2 eps in the distance and 4 eps after CSLS, for either of the two). Exact ties are decided too:
    equal rows give equal scores in any arithmetic."""
    srt = np.sort(ref["dist"], 1)
    if srt.shape[1] < 5:
        return np.ones((srt.shape[0],), bool)
    gap = srt[:, 4] - srt[:, 2]
    return (gap > 8.0 * eps) | (gap == 0)


def assert_equal_to_oracle(res, ref: dict, csls: bool, want_top3: bool, top3_rows=None, out: dict | None = None) -> None:
    """Ranks, g, nv1 / nv2 (no unverified neighbourhood), the prediction ids and Hits@k / MR / MRR bit for bit."""
    np.testing.assert_array_equal(res.rank_l2r.cpu().numpy(), ref["rank_l2r"])
    np.testing.assert_array_equal(res.rank_r2l.cpu().numpy(), ref["rank_r2l"])
    np.testing.assert_array_equal(res.g.cpu().numpy(), ref["g"])
    if csls:
        np.testing.assert_array_equal(res.nv1.cpu().numpy(), ref["nv1"])
        np.testing.assert_array_equal(res.nv2.cpu().numpy(), ref["nv2"])
        assert all(v.get("unverified", 0) == 0 for v in res.info.get("neighbourhoods", {}).values()), res.info
    if want_top3:
        got = res.top3_idx.cpu().numpy()
        rows = np.ones((got.shape[0],), bool) if top3_rows is None else top3_rows
        np.testing.assert_array_equal(got[rows], ref["top3"][rows])
    for side in ("l2r", "r2l"):
        o = oracle.metrics(ref[f"rank_{side}"])
        for m in (evaluate.metrics_from_ranks(getattr(res, f"rank_{side}")),) + ((out[side],) if out is not None else ()):
            assert m.mr == o["mr"] and m.mrr == o["mrr"] and np.array_equal(m.acc, o["acc"]), (side, m, o)
