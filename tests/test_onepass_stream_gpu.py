"""The one-pass evaluation sweep (sim_kernel<EpiOnePass>) streams exactly the elements its exact fp32 tests accept: its
fp16x2 pre-filter may flag more, never less, and the warp-aggregated appends lose or duplicate nothing. S is materialised
with sim_kernel<EpiWrite> (the same mainloop, the same bits) and the two streams are rebuilt in torch."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from oracle import oracle
from snag_b200 import evaluate, ops

pytestmark = pytest.mark.gpu

N, D, K = 20000, 1200, 10


def _capture_constants(monkeypatch, X, Y, xn, yn, n):
    """Run the one-pass evaluation (forced on at this size) and return the arguments its sweep was launched with."""
    monkeypatch.setattr(evaluate, "TWO_SWEEP_MIN_N", 16384)
    calls = []
    orig = ops.eval_onepass

    def spy(*a, **kw):
        calls.append((a, kw))
        return orig(*a, **kw)

    monkeypatch.setattr(ops, "eval_onepass", spy)
    res = evaluate.align_ranks(X, Y, xn, yn, n, K, True, one_pass=True)
    assert len(calls) == 1 and res.info["one_pass"] is not None
    return calls[0]


def _decode(stream, rows, cnt, n_cols):
    cap = stream.shape[1]
    cnt = cnt.long()
    keep = torch.arange(cap, device=stream.device)[None, :] < cnt.clamp(max=cap)[:, None]
    s = stream[keep]
    col = (s & 0xFFFFFFFF).long()
    bits = (s >> 32).to(torch.int32)
    key = rows[keep].long() * n_cols + col
    order = torch.argsort(key)
    return key[order], bits[order]


def _expected(S, mask, vals, n_cols):
    r, c = mask.nonzero(as_tuple=True)
    key = r.long() * n_cols + c.long()
    bits = vals[mask].view(torch.int32)
    order = torch.argsort(key)                     # nonzero is row-major already; sorted for symmetry with _decode
    return key[order], bits[order]


def _check_streams(X, Y, xn, yn, n, args, small_caps=False):
    (X_, Y_, xn_, yn_, n1, n2, colthr, colb, cta_cap, rowthr, rk_r, rk_rp, rk_c, rk_cp, rk_cap, *rest) = args
    if small_caps:
        cta_cap, rk_cap = 257, 129
    out = ops.eval_onepass(X, Y, xn, yn, n1, n2, colthr, colb, cta_cap, rowthr, rk_r, rk_rp, rk_c, rk_cp, rk_cap, *rest)
    _, _, stream, stream_row, stream_cnt, rk_stream, rk_stream_row, rk_cnt = out
    S = ops.sim_write(X, Y, None, None, n1, n2, 0)
    # rank candidates: s > min(R_i + C_j, R'_i + C'_j), the tensor-core s streamed
    thr = torch.minimum(rk_r[:n1, None] + rk_c[None, :n2], rk_rp[:n1, None] + rk_cp[None, :n2])
    want_rk = _expected(S, S > thr, S, n2)
    del thr
    # column candidates: s > xn_i / 2 + b_j and c = 1 - max((xn_i + yn_j) - 2 s, 0) >= colthr_j, c streamed
    want_col_mask = S > (0.5 * xn[:n1, None] + colb[None, :n2])
    c = 1.0 - torch.clamp((xn[:n1, None] + yn[None, :n2]) - 2.0 * S, min=0.0)
    want_col_mask &= c >= colthr[None, :n2]
    want_col = _expected(S, want_col_mask, c, n2)
    del S, c, want_col_mask
    for name, got_args, want, cap in (("rank", (rk_stream, rk_stream_row, rk_cnt), want_rk, rk_cap),
                                      ("column", (stream, stream_row, stream_cnt), want_col, cta_cap)):
        key, bits = _decode(*got_args, n2)
        cnt = got_args[2].long()
        if not small_caps:
            assert int(cnt.max()) <= cap, f"{name} stream overflowed"
            assert torch.equal(key, want[0]), f"{name} stream: {key.numel()} entries, expected {want[0].numel()}"
            assert torch.equal(bits, want[1]), f"{name} stream values differ"
        else:
            # overflow: every CTA that ran out reports a count above its capacity (the counter saturates a little
            # above it, it does not wrap), and what was stored is a duplicate-free subset of the exact set
            assert int(cnt.max()) > cap and int(cnt.max()) <= cap + 32 * 8, (name, int(cnt.max()))
            assert torch.unique(key).numel() == key.numel()
            pos = torch.searchsorted(want[0], key)
            assert bool((pos < want[0].numel()).all())
            assert torch.equal(want[0][pos], key) and torch.equal(want[1][pos], bits), name
    return want_rk[0].numel(), want_col[0].numel()


def _bench_rows(n, dev, scale=None):
    import bench
    emb, left, right = bench.synth_tables(n, D, 6.0, dev)
    if scale is None:
        X, xn = ops.prep_bf16(emb, left, True)
        Y, yn = ops.prep_bf16(emb, right, True)
        return X, Y, xn, yn
    # rows off unit norm by as much as the fp16x2 pre-filter is allowed to take (HALF_PREFILTER_NORM2_MAX)
    x = torch.nn.functional.normalize(emb[left], dim=1) * scale(n, dev)[:, None]
    y = torch.nn.functional.normalize(emb[right], dim=1) * scale(n, dev)[:, None]
    X, xn = ops.prep_bf16(x, None, False)
    Y, yn = ops.prep_bf16(y, None, False)
    assert float(torch.maximum(xn.max(), yn.max())) <= ops.HALF_PREFILTER_NORM2_MAX
    return X, Y, xn, yn


def _fp16_boundaries(v):
    """Move every constant onto an fp16 rounding boundary: alternately an fp16 value, one fp32 ulp above it, the
    midpoint to the next fp16 value up, and one fp32 ulp below that midpoint."""
    h = v.half().float()
    ulp = torch.exp2(torch.floor(torch.log2(h.abs().clamp(min=2.0 ** -14))) - 10.0)
    mid = h + 0.5 * ulp
    sel = torch.arange(v.numel(), device=v.device) % 4
    up = torch.nextafter(h, torch.full_like(h, float("inf")))
    below_mid = torch.nextafter(mid, torch.full_like(mid, float("-inf")))
    out = torch.where(sel == 0, h, torch.where(sel == 1, up, torch.where(sel == 2, mid, below_mid)))
    return torch.where(torch.isfinite(v), out, v).contiguous()


@pytest.mark.parametrize("variant", ["bench", "fp16_boundaries", "off_unit_norm"])
def test_prefilter_never_drops_an_element(cuda_device, monkeypatch, variant):
    dev = cuda_device
    if variant == "off_unit_norm":
        def scale(n, d):                           # squared norms spread over [0.96, 1.045]
            g = torch.Generator(device="cpu").manual_seed(5)
            return (0.96 + 0.085 * torch.rand((n,), generator=g)).sqrt().to(d)
        X, Y, xn, yn = _bench_rows(N, dev, scale)
    else:
        X, Y, xn, yn = _bench_rows(N, dev)
    args, kw = _capture_constants(monkeypatch, X, Y, xn, yn, N)
    args = list(args)
    if variant == "fp16_boundaries":
        for i in (7, 10, 11, 12, 13):              # colb, rk_r, rk_rp, rk_c, rk_cp
            args[i] = _fp16_boundaries(args[i])
    n_rk, n_col = _check_streams(X, Y, xn, yn, N, args)
    assert n_rk > 1000 and n_col > 1000, (n_rk, n_col)      # the sets are not trivially empty
    _check_streams(X, Y, xn, yn, N, args, small_caps=True)


@pytest.mark.parametrize("world", [1, 4])
def test_one_pass_c1_shape_equals_oracle(cuda_device, monkeypatch, world):
    """The one-pass evaluation forced on at the C1 shape (10 500 pairs, D = 1200, k = 10): nv1, nv2, g and both rank
    vectors bit-identical to the oracle, on one and on four simulated ranks."""
    monkeypatch.setattr(evaluate, "TWO_SWEEP_MIN_N", 8192)
    oracle.set_threads()
    n, d, k = 10500, 1200, 10
    rng = np.random.RandomState(3408)
    centres = rng.randn(64, d).astype(np.float32)
    x = rng.randn(n, d).astype(np.float32) + centres[rng.randint(0, 64, n)]
    y = x + np.float32(8.0) * rng.randn(n, d).astype(np.float32)
    x, y = oracle.bf16_round(oracle.normalize_rows(x)), oracle.bf16_round(oracle.normalize_rows(y))
    X, xn = ops.prep_bf16(torch.from_numpy(x).to(cuda_device), None, normalize=False)
    Y, yn = ops.prep_bf16(torch.from_numpy(y).to(cuda_device), None, normalize=False)
    ref = oracle.align_eval(x, y, True, k)
    res = evaluate.simulate_sharded(
        lambda r: evaluate._align_ranks_steps(ops, X, Y, xn, yn, n, k, True, False, world, r, one_pass=True), world)
    for mr in res:
        assert mr.info["one_pass"] is not None and mr.info["one_pass"]["fallback"] is None, mr.info["one_pass"]
    out = res[0]
    for key in ("nv1", "nv2", "g", "rank_l2r", "rank_r2l"):
        np.testing.assert_array_equal(getattr(out, key).cpu().numpy(), ref[key], err_msg=key)
