"""GPU: the three fused evaluation routes — bf16 (`ops`), fp32 (`fp32`, split operands) and --distance 1 (`l1`) — at the
edges of tests/eval_edges.py, bit for bit against the oracle: ragged n around the 128-row and 256-column tiles, widths
across Dpad and the prologue's register windows, CSLS on and off with k up to n, sharded runs whose trailing ranks own
one target or none, degenerate tables (zero rows, repeated rows, one row repeated, one-hot rows) and n at the size where
the two-sweep path takes over. Then the prologue kernels (prep_bf16, fp32.prep, icl_stack_prep, l1.prep) against an
fp64 normalisation with a bound derived from their arithmetic, bitwise invariants and exact rescalings."""
from __future__ import annotations

import math

import numpy as np
import pytest
import torch

from oracle import oracle
from snag_b200 import _lib, evaluate, fp32, l1, ops
from tests import eval_edges as ee

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _oracle_threads():
    oracle.set_threads()


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(dev)


def _pairs(x, y, dev):
    """final_emb = [x ; y] and the pair ids of evaluate_alignment*."""
    n = x.shape[0]
    return _t(np.concatenate([x, y], 0), dev), torch.arange(0, n, device=dev), torch.arange(n, 2 * n, device=dev)


def _steps(be, X, Y, xn, yn, n, k, csls, top3, world, **kw):
    return evaluate.simulate_sharded(
        lambda r: evaluate._align_ranks_steps(be, X, Y, xn, yn, n, k, csls, top3, world, r, **kw), world)


def _evaluate(route, path, x, y, csls, k, top3, dev, world=1):
    """(results of every rank, metrics dict of the entry point or None, the rows the oracle must see, band eps in s)."""
    n, d = x.shape
    out = None
    if route == "bf16":
        x, y = oracle.bf16_round(x), oracle.bf16_round(y)
        eps = ops.tc_margin(evaluate.round_up(d, 64))
        if path == "graph":
            out = evaluate.evaluate_alignment(*_pairs(x, y, dev), csls=csls, csls_k=k, want_top3=top3, normalize=False,
                                              graph=True)
            return [out["ranks"]], out, x, y, eps
        X, xn = ops.prep_bf16(_t(x, dev), None, normalize=False)
        Y, yn = ops.prep_bf16(_t(y, dev), None, normalize=False)
        if path == "lazy":
            res = evaluate._align_ranks_lazy(ops, X, Y, xn, yn, n, k, csls, top3)
            if res is None:                  # an assumption of the sync-free path failed: what align_ranks does next
                res = evaluate.align_ranks(X, Y, xn, yn, n, k, csls, top3, lazy=False)
            return [res], None, x, y, eps
        return _steps(ops, X, Y, xn, yn, n, k, csls, top3, world), None, x, y, eps
    if route == "fp32":
        eps = fp32.tc_margin(evaluate.round_up(d, 64))
        if path == "entry":
            out = evaluate.evaluate_alignment(*_pairs(x, y, dev), csls=csls, csls_k=k, want_top3=top3, normalize=False,
                                              precision="fp32")
            return [out["ranks"]], out, x, y, eps
        X, xn = fp32.prep(_t(x, dev), None, False, 0)
        Y, yn = fp32.prep(_t(y, dev), None, False, 1)
        return _steps(fp32, X, Y, xn, yn, n, k, csls, top3, world), None, x, y, eps
    emb, left, right = _pairs(x, y, dev)
    fe = torch.nn.functional.normalize(emb)                          # main.py:379, as evaluate_alignment_l1 does
    xs, ys = fe[:n].cpu().numpy(), fe[n:].cpu().numpy()
    if path == "entry":
        out = evaluate.evaluate_alignment_l1(emb, left, right, csls=csls, csls_k=k, want_top3=top3)
        return [out["ranks"]], out, xs, ys, 0.0
    X, xn = l1.prep(fe, left)
    Y, yn = l1.prep(fe, right)
    return _steps(l1, X, Y, xn, yn, n, k, csls, top3, world, two_sweep=False), None, xs, ys, 0.0


def _oracle(route, x, y, csls, k, top3):
    if route == "l1":
        return oracle.align_eval_l1(x, y, csls, k)
    return oracle.align_eval(x, y, csls, k, want_dist=top3)


def _check(route, res, out, ref, csls, top3, eps):
    # the L1 route rescans every row its 4 candidates cannot vouch for: its prediction ids are exact on every row
    rows = ee.top3_checkable(ref, eps) if top3 and route != "l1" else None
    if rows is not None:
        assert rows.mean() >= 0.9, rows.mean()
    ee.assert_equal_to_oracle(res, ref, csls, top3, rows, None if out is None else {"l2r": out["l2r"], "r2l": out["r2l"]})


def _ids(cases):
    return ["-".join(str(v) for v in c) for c in cases]


# ------------------------------------------------------------------------------------------------ the edge table
_EDGES = [(route,) + c for route in ee.ROUTES for c in ee.edge_cases(route)]


@pytest.mark.parametrize("route,n,d,csls,k,want_top3,path", _EDGES, ids=_ids(_EDGES))
def test_edge_table_against_the_oracle(cuda_device, route, n, d, csls, k, want_top3, path):
    x, y = ee.clustered(n, d, 1.0, n + d)
    many, out, xo, yo, eps = _evaluate(route, path, x, y, csls, k, want_top3, cuda_device)
    ref = _oracle(route, xo, yo, csls, k, want_top3)
    _check(route, many[0], out, ref, csls, want_top3, eps)
    if path == "graph":
        assert many[0].info.get("cuda_graph") is True
    if route == "fp32" and path == "entry":
        assert many[0].info["precision"] == "fp32"
    if route == "l1" and path == "entry":
        assert many[0].info["distance"] == 1 and not many[0].info.get("materialised")


@pytest.mark.parametrize("route", ee.ROUTES)
def test_neighbourhoods_larger_than_n_are_refused(cuda_device, route):
    """k > n raises in the reference (torch.topk): every entry point refuses it the same way, before any kernel."""
    x, y = ee.clustered(2, 8, 1.0, 2)
    emb, left, right = _pairs(x, y, cuda_device)
    call = {"bf16": lambda **kw: evaluate.evaluate_alignment(emb, left, right, **kw),
            "fp32": lambda **kw: evaluate.evaluate_alignment(emb, left, right, precision="fp32", **kw),
            "l1": lambda **kw: evaluate.evaluate_alignment_l1(emb, left, right, **kw)}[route]
    for k in (3, 0):
        with pytest.raises(ValueError):
            call(csls=True, csls_k=k)
    if route == "bf16":
        X, xn = ops.prep_bf16(_t(x, cuda_device), None, normalize=False)
        with pytest.raises(ValueError):
            evaluate.align_ranks(X, X, xn, xn, 2, 3, True)
        with pytest.raises(_lib.SnagError):
            evaluate.align_ranks(X, X, xn, xn, 2, 17, True)


# ------------------------------------------------------------------------------------------------ sharding
_SHARDED = [(route,) + c for route in ee.ROUTES for c in ee.sharded_cases(route)]


@pytest.mark.parametrize("route,n,d,world,csls,k", _SHARDED, ids=_ids(_SHARDED))
def test_sharded_with_empty_trailing_ranks(cuda_device, route, n, d, world, csls, k):
    sizes = ee.shard_sizes(n, world)
    assert sum(sizes) == n and min(sizes) <= 1, sizes             # a rank owns one target or none
    x, y = ee.clustered(n, d, 1.0, 7 * n + world)
    many, _, xo, yo, eps = _evaluate(route, "generator", x, y, csls, k, True, cuda_device, world)
    ref = _oracle(route, xo, yo, csls, k, True)
    assert len(many) == world
    for r in many:                                                  # every rank ends with the full result
        assert r.info["shard"] == evaluate.shard_bounds(n, world, r.info["rank"])
        _check(route, r, None, ref, csls, True, eps)


# ------------------------------------------------------------------------------------------------ degenerate tables
_DEGENERATE = [(route,) + c for route in ee.ROUTES for c in ee.degenerate_cases(route)]


@pytest.mark.parametrize("route,table,n,d", _DEGENERATE, ids=_ids(_DEGENERATE))
def test_degenerate_tables(cuda_device, monkeypatch, route, table, n, d):
    paths = ee.PATHS[route]
    path = paths[(ee.DEGENERATE.index(table) + (n > 257)) % len(paths)]
    all_ties = table == "one_row"
    if all_ties:
        # n (n - 1) elements tie with their ground truth: a first list smaller than that must overflow and grow
        monkeypatch.setattr(ops, "RANK_BAND_MIN_CAP", 4096)
        monkeypatch.setattr(ops, "RANK_BAND_PER_ROW", 0)
        monkeypatch.setattr(l1, "BAND_MIN_CAP", 4096)
        monkeypatch.setattr(l1, "BAND_PER_ROW", 0)
    first_cap = (max(l1.BAND_MIN_CAP, l1.BAND_PER_ROW * 2 * n) if route == "l1" else
                 max(ops.RANK_BAND_MIN_CAP, ops.RANK_BAND_PER_ROW * 2 * n))
    x, y = ee.degenerate(table, n, d, n + d)
    many, out, xo, yo, eps = _evaluate(route, path, x, y, True, 10, True, cuda_device)
    res = many[0]
    ref = _oracle(route, xo, yo, True, 10, True)
    _check(route, res, out, ref, True, True, eps)
    if table == "zero_rows":
        assert (xo == 0).all(1).any() and (yo == 0).all(1).any()
    if all_ties:
        np.testing.assert_array_equal(ref["rank_l2r"], np.arange(n))        # the stable order: lower index first
        np.testing.assert_array_equal(res.top3_idx.cpu().numpy(), np.tile(np.arange(3), (n, 1)))
        rs = res.info["rank_sweep"]
        # the deferral list overflowed its first size and the sweep was redone with a larger one
        assert rs["mode"] == "band" and rs["deferred"] > first_cap and rs["cap"] >= rs["deferred"], rs
    elif path == "graph":
        assert res.info.get("cuda_graph") is True


# ------------------------------------------------------------------------------------------------ the switch point
@pytest.fixture(scope="module")
def switch_problem():
    n, d = evaluate.TWO_SWEEP_MIN_N, 64
    x, y = ee.clustered(n, d, 4.0, 3411)
    return x, y


@pytest.mark.parametrize("route", ["bf16", "fp32"])
def test_two_sweep_switch_point(cuda_device, switch_problem, route):
    """n = TWO_SWEEP_MIN_N exactly takes the two-sweep path (the sample pre-passes), one-pass or not."""
    x, y = switch_problem
    n, k = x.shape[0], 10
    assert evaluate.two_sweep_plan(n, k) is not None and evaluate.two_sweep_plan(n - 1, k) is None
    if route == "bf16":
        x, y = oracle.bf16_round(x), oracle.bf16_round(y)
        X, xn = ops.prep_bf16(_t(x, cuda_device), None, normalize=False)
        Y, yn = ops.prep_bf16(_t(y, cuda_device), None, normalize=False)
    else:
        X, xn = fp32.prep(_t(x, cuda_device), None, False, 0)
        Y, yn = fp32.prep(_t(y, cuda_device), None, False, 1)
    ref = oracle.align_eval_stream(x, y, True, k, 2048)
    for one_pass, kernel in ((True, "sim_kernel<EpiOnePass>"), (False, "sim_kernel<EpiRowColTopK>")):
        sweeps = []
        ops.SWEEP_EVENT_SINK = sweeps
        try:
            if route == "bf16":
                res = evaluate.align_ranks(X, Y, xn, yn, n, k, True, one_pass=one_pass)
            else:
                res = _steps(fp32, X, Y, xn, yn, n, k, True, False, 1, one_pass=one_pass)[0]
        finally:
            ops.SWEEP_EVENT_SINK = None
        names = [nm for nm, *_ in sweeps]
        assert kernel in names, names
        if not one_pass:
            assert "sim_kernel<EpiOnePass>" not in names
        ee.assert_equal_to_oracle(res, ref, True, False)            # exact whatever the one-pass evaluation fell back to


# ------------------------------------------------------------------------------------------------ prologue kernels
P_WIDTHS = (1, 3, 4, 63, 64, 65, 97, 508, 512, 516, 2044, 2048, 2052, 4096)
U = 2.0 ** -24                 # fp32 unit roundoff
U_BF16 = 2.0 ** -8             # bf16 unit roundoff (8 significant bits)


def _lane_chain(d: int, vec4: bool) -> int:
    """Length L of one lane's fp32 FMA chain of squares: float4 path 4 per float4, lanes 128 columns apart; scalar path
    one per column, lanes 32 apart."""
    return 4 * math.ceil(d / 128) if vec4 else math.ceil(d / 32)


def _normalise_bound(d: int, vec4: bool) -> float:
    """Relative error bound of a normalised element z = x / max(||x||, 1e-12) against fp64:
      ss  = each lane's chain of L fp32 FMAs (one rounding each, all terms >= 0), then 5 butterfly additions:
            ss~ = ss (1 + t), |t| <= gamma(L + 5) = (L + 5) u / (1 - (L + 5) u);
      sqrtf halves that and adds one rounding, __fdiv_rn adds one more:
            z~ = z (1 + d2) / ((1 + t)^(1/2) (1 + d1)), so |z~ / z - 1| <= ((L + 5) / 2 + 2) u + O(u^2).
    The second-order terms are below (L + 7)^2 u^2, under 2^-8 of the first-order bound for L <= 128: bounded by that
    factor. A clamped denominator (||x|| < 1e-12) leaves the division's rounding alone, inside the same bound."""
    L = _lane_chain(d, vec4)
    return ((L + 5) / 2 + 2) * U * (1 + 2.0 ** -8)


def _misaligned(t: torch.Tensor) -> torch.Tensor:
    """A contiguous copy of t whose base is 4 bytes past a 16-byte boundary: the prologues take their scalar path."""
    buf = torch.empty((t.numel() + 4,), dtype=t.dtype, device=t.device)
    v = buf[1:1 + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 == 4
    return v


def _paths(d):
    return (True, False) if d % 4 == 0 else (False,)


def _prologue_table(d: int, seed: int) -> np.ndarray:
    """Rows of varied norms: a zero row, a row below the 1e-12 clamp, a one-hot row, wide dynamic range, random."""
    rng = np.random.RandomState(seed)
    e = (rng.randn(96, d) * rng.rand(96, 1) * 5).astype(np.float32)
    e[3] = 0.0
    e[5] = (rng.randn(d) * 1e-14 / math.sqrt(d)).astype(np.float32)
    e[7] = 0.0
    e[7, rng.randint(d)] = -3.0
    e[11] *= np.exp2(rng.randint(-30, 4, d)).astype(np.float32)
    return e


def _indices(dev):
    rng = np.random.RandomState(1)
    return {"duplicates": torch.from_numpy(np.concatenate([[3, 5, 7, 11], rng.randint(0, 96, 60), [3, 3]])).to(dev),
            "reversed": torch.arange(95, -1, -1, device=dev),
            "single": torch.tensor([5], device=dev)}


def _fp64_normalised(rows: np.ndarray) -> np.ndarray:
    r = rows.astype(np.float64)
    return r / np.maximum(np.sqrt((r * r).sum(1)), np.float64(np.float32(1e-12)))[:, None]


def _bf16_bits(t: torch.Tensor) -> np.ndarray:
    return t.contiguous().view(torch.int16).cpu().numpy()


def _rn_bf16(a: np.ndarray) -> np.ndarray:
    return oracle.bf16_round(np.ascontiguousarray(a, np.float32))


def _junk_pool(shapes, dev):
    """Fill and release blocks of the sizes the next allocations will have ((shape, dtype) pairs), so that output a
    prologue fails to write (padding) reads as NaN junk rather than as the zeros of fresh device memory."""
    for s, dtype in shapes:
        torch.full(s, float("nan"), dtype=dtype, device=dev)


@pytest.mark.parametrize("d", P_WIDTHS)
def test_prologues_against_fp64(cuda_device, d):
    emb_h = _prologue_table(d, d)
    dpad = evaluate.round_up(d, 64)
    worst = {True: 0.0, False: 0.0}          # largest error / bound of the fp32 rows, per path
    for vec4 in _paths(d):
        emb = _t(emb_h, cuda_device)
        emb = emb if vec4 else _misaligned(emb)
        tol = _normalise_bound(d, vec4)
        for name, idx in _indices(cuda_device).items():
            src = emb_h[idx.cpu().numpy()]
            z = _fp64_normalised(src)
            n = src.shape[0]
            for normalize in (True, False):
                want = z if normalize else src.astype(np.float64)
                splits = []
                for side in (0, 1):
                    _junk_pool([((n, dpad), torch.float32), ((n, 3 * dpad), torch.bfloat16)], cuda_device)
                    S, nrm = fp32.prep(emb, idx, normalize, side)
                    rows = S.rows.cpu().numpy()
                    assert not rows[:, d:].any(), (name, side)                       # zero padded columns
                    if normalize:
                        ratio = float((np.abs(rows[:, :d] - z) / np.maximum(tol * np.abs(z), 1e-300)).max())
                        worst[vec4] = max(worst[vec4], ratio)
                        assert ratio <= 1.0, (name, side, vec4, ratio)
                    else:
                        np.testing.assert_array_equal(rows[:, :d], src)
                    np.testing.assert_array_equal(nrm.cpu().numpy(), oracle.norm2(rows[:, :d]))
                    h = _rn_bf16(rows)
                    m = _rn_bf16(rows - h)
                    sp = S.split.float().cpu().numpy()
                    parts = (h, m, h) if side else (m, h, h)                         # [h | m | h] targets, [m | h | h] sources
                    for p, want_p in enumerate(parts):
                        np.testing.assert_array_equal(sp[:, p * dpad:(p + 1) * dpad], want_p)
                    splits.append(rows)
                np.testing.assert_array_equal(splits[0], splits[1])
                out = torch.full((n, dpad), float("nan"), dtype=torch.bfloat16, device=cuda_device)
                B, bn = ops.prep_bf16(emb, idx, normalize, out=out)
                assert B.data_ptr() == out.data_ptr()
                b = B.float().cpu().numpy()
                assert not b[:, d:].any()                                             # padding written over the junk
                np.testing.assert_array_equal(b, _rn_bf16(splits[0]))                 # h = RN-bf16 of the fp32 rows
                err = np.abs(b[:, :d] - want)
                assert (err <= (tol if normalize else 0.0) * np.abs(want) + U_BF16 * np.abs(want) * (1 + tol)).all()
                np.testing.assert_array_equal(bn.cpu().numpy(), oracle.norm2(b[:, :d]))
                if not normalize:
                    np.testing.assert_array_equal(b[:, :d], _rn_bf16(src))
                zero = (src == 0).all(1)
                assert not b[zero].any() and not bn.cpu().numpy()[zero].any()
                Xl, xnl = l1.prep(emb, idx)
                assert Xl.shape == (n, evaluate.round_up(d, 8))
                xl = Xl.cpu().numpy()
                np.testing.assert_array_equal(xl[:, :d], src)
                assert not xl[:, d:].any()
                np.testing.assert_array_equal(xnl.cpu().numpy(), np.abs(src.astype(np.float64)).sum(1).astype(np.float32))
    print(f"\n[prologue D={d}] worst error / bound: float4 path {worst[True]:.3f}, scalar path {worst[False]:.3f}")


def test_icl_stack_prep_two_launches_of_mixed_widths(cuda_device):
    """17 tables (two launches of at most MANY_MAX), narrow and wide in each: every part is prep_bf16 of its indices,
    rows B..Bp of every part are zero and the third part repeats the first, on the float4 and the scalar path."""
    widths = P_WIDTHS + (1, 516, 4096)
    assert len(widths) == ops.MANY_MAX + 1
    tables = [_prologue_table(d, 100 + d) for d in widths]
    idx = _indices(cuda_device)
    pairs = {"duplicates/reversed": (idx["duplicates"][:60].contiguous(), idx["reversed"][:60].contiguous()),
             "single": (idx["single"], idx["single"])}
    for aligned in (True, False):
        embs = [_t(e, cuda_device) for e in tables]
        if not aligned:
            embs = [_misaligned(e) for e in embs]
        for tag, (il, ir) in pairs.items():
            B, Bp = il.numel(), 256
            for normalize in (True, False):
                _junk_pool([((3 * Bp, evaluate.round_up(d, 64)), torch.bfloat16) for d in widths], cuda_device)
                outs = ops.icl_stack_prep(embs, il, ir, Bp, normalize)
                for e, eh, d, S3 in zip(embs, tables, widths, outs):
                    dpad = evaluate.round_up(d, 64)
                    assert S3.shape == (3 * Bp, dpad)
                    s = _bf16_bits(S3)
                    a, b = ops.prep_bf16(e, il, normalize)[0], ops.prep_bf16(e, ir, normalize)[0]
                    np.testing.assert_array_equal(s[:B], _bf16_bits(a), err_msg=f"{tag} D={d}")
                    np.testing.assert_array_equal(s[Bp:Bp + B], _bf16_bits(b), err_msg=f"{tag} D={d}")
                    np.testing.assert_array_equal(s[2 * Bp:], s[:Bp])
                    for p in range(3):
                        assert not s[p * Bp + B:(p + 1) * Bp].any(), (tag, d, p)
                    if not normalize:
                        np.testing.assert_array_equal(S3[:B].float().cpu().numpy()[:, :d], _rn_bf16(eh[il.cpu().numpy()]))


@pytest.mark.parametrize("d", P_WIDTHS)
def test_prologues_are_scale_invariant(cuda_device, d):
    """Rows scaled by 2^k normalise to the same bits: the sums of squares scale by 2^2k exactly, the square root by 2^k
    and the division cancels it. The rows are built so that every square stays normal and every norm above the clamp
    (||x|| ~ 2^12, elements bounded away from zero)."""
    rng = np.random.RandomState(d)
    base = (np.where(rng.rand(64, d) < 0.5, -1.0, 1.0) * (0.5 + rng.rand(64, d))).astype(np.float32)
    base = (oracle.normalize_rows(base) * np.float32(4096.0)).astype(np.float32)
    base[9] = 0.0
    ids = rng.randint(0, 64, 80)
    ids[[0, 50]] = 9
    idx = torch.from_numpy(ids).to(cuda_device)
    il, ir = idx[:40].contiguous(), idx[40:].contiguous()

    def outputs(e):
        t = _t(e, cuda_device)
        res = []
        for vec4 in _paths(d):
            tt = t if vec4 else _misaligned(t)
            S0, n0 = fp32.prep(tt, idx, True, 0)
            S1, n1 = fp32.prep(tt, idx, True, 1)
            B, bn = ops.prep_bf16(tt, idx, True)
            S3 = ops.icl_stack_prep([tt], il, ir, 256, True)[0]
            res += [S0.rows.cpu().numpy().view(np.uint32), _bf16_bits(S0.split), _bf16_bits(S1.split), n0.cpu().numpy(),
                    n1.cpu().numpy(), _bf16_bits(B), bn.cpu().numpy(), _bf16_bits(S3)]
        return res

    want = outputs(base)
    zero = ids == 9
    assert not want[0][zero].any() and not want[3][zero].any() and not want[6][zero].any()   # zero rows: zeros, norm2 = 0
    for k in (-50, -20, 20, 50):
        got = outputs((base * np.float32(2.0 ** k)).astype(np.float32))
        for a, b in zip(got, want):
            np.testing.assert_array_equal(a, b, err_msg=f"2^{k}")
