"""GPU: the fp32 evaluation (evaluate_alignment(precision="fp32"), snag_b200.fp32) on UNROUNDED fp32 rows — the
prologue bit for bit, the fp32 canonical kernels, every output bit-equal to oracle.align_eval at the baseline sizes
(1, 2 and 8 ranks) and above TWO_SWEEP_MIN_N (one-pass and two-sweep paths, 1 and 4 ranks), bf16-representable goldens
where the fp32 mode must equal the bf16 mode, and the measurement of the split operands' tensor-core error that fixes
fp32.FP32_TC_DOT_ERR_PER_K."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from oracle import oracle
from snag_b200 import evaluate, fp32, ops
from tests.conftest import golden_names, load_golden

pytestmark = pytest.mark.gpu


def _clustered(n, d, sigma, seed):
    """The baseline tests' generator (64 cluster centres, noisy copies as targets), normalised but NOT rounded to bf16."""
    rng = np.random.RandomState(seed)
    centres = rng.randn(64, d).astype(np.float32)
    x = rng.randn(n, d).astype(np.float32) + centres[rng.randint(0, 64, n)]
    y = x + np.float32(sigma) * rng.randn(n, d).astype(np.float32)
    return oracle.normalize_rows(x), oracle.normalize_rows(y)


def _prep(x, y, dev):
    X, xn = fp32.prep(torch.from_numpy(np.ascontiguousarray(x)).to(dev), None, False, 0)
    Y, yn = fp32.prep(torch.from_numpy(np.ascontiguousarray(y)).to(dev), None, False, 1)
    return X, Y, xn, yn


def _run(X, Y, xn, yn, n, k, csls, want_top3=False, world=1, **kw):
    many = evaluate.simulate_sharded(
        lambda r: evaluate._align_ranks_steps(fp32, X, Y, xn, yn, n, k, csls, want_top3, world, r, **kw), world)
    return many


def _assert_equal_to_oracle(res, ref, csls):
    if csls:
        np.testing.assert_array_equal(res.nv1.cpu().numpy(), ref["nv1"])
        np.testing.assert_array_equal(res.nv2.cpu().numpy(), ref["nv2"])
        info = res.info["neighbourhoods"]
        assert info["rows"]["unverified"] == 0 and info["cols"]["unverified"] == 0
    np.testing.assert_array_equal(res.g.cpu().numpy(), ref["g"])
    np.testing.assert_array_equal(res.rank_l2r.cpu().numpy(), ref["rank_l2r"])
    np.testing.assert_array_equal(res.rank_r2l.cpu().numpy(), ref["rank_r2l"])
    for side, ranks in (("l2r", res.rank_l2r), ("r2l", res.rank_r2l)):
        m = evaluate.metrics_from_ranks(ranks)
        o = oracle.metrics(ref[f"rank_{side}"])
        assert m.mr == o["mr"] and m.mrr == o["mrr"] and np.array_equal(m.acc, o["acc"])


def _bf16_bits(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(torch.int16)


@pytest.mark.parametrize("d", [300, 97, 1200])            # float4 path (D % 4 == 0) and scalar path (D = 97)
def test_prologue_bits(cuda_device, d):
    rng = np.random.RandomState(d)
    emb = torch.from_numpy((rng.randn(900, d) * rng.rand(900, 1) * 5).astype(np.float32)).to(cuda_device)
    idx = torch.from_numpy(rng.randint(0, 900, 700)).to(cuda_device)
    dpad = evaluate.round_up(d, 64)
    for side in (0, 1):
        S, xn = fp32.prep(emb, idx, True, side)
        Xb, _ = ops.prep_bf16(emb, idx, True)
        rows, split = S.rows, S.split
        h = split[:, 2 * dpad:]
        hs = split[:, :dpad] if side else split[:, dpad:2 * dpad]
        m = split[:, dpad:2 * dpad] if side else split[:, :dpad]
        assert torch.equal(_bf16_bits(h), _bf16_bits(Xb)) and torch.equal(_bf16_bits(hs), _bf16_bits(Xb))
        assert torch.equal(_bf16_bits(rows.to(torch.bfloat16)), _bf16_bits(Xb))        # h = bf16(x)
        assert torch.equal(_bf16_bits(m), _bf16_bits((rows - h.float()).to(torch.bfloat16)))
        assert torch.equal(rows[:, d:], torch.zeros_like(rows[:, d:]))
        np.testing.assert_array_equal(xn.cpu().numpy(), oracle.norm2(rows[:, :d].cpu().numpy()))
        # the fp32 rows are F.normalize's values
        want = torch.nn.functional.normalize(emb.index_select(0, idx), dim=1)
        assert float((rows[:, :d] - want).abs().max()) <= 2e-7
    # normalize=False: the host rows themselves, bit for bit
    S, xn = fp32.prep(emb, None, False, 0)
    assert torch.equal(S.rows[:, :d], emb)
    np.testing.assert_array_equal(xn.cpu().numpy(), oracle.norm2(emb.cpu().numpy()))


def test_pairs_dot_f32_is_the_oracle_dot(cuda_device):
    x, y = _clustered(600, 1200, 8.0, 5)
    X, Y, _, _ = _prep(x, y, cuda_device)
    rng = np.random.RandomState(2)
    ri, ci = rng.randint(0, 600, 5000).astype(np.int32), rng.randint(0, 600, 5000).astype(np.int32)
    got = fp32.pairs_dot(X, Y, torch.from_numpy(ri).to(cuda_device), torch.from_numpy(ci).to(cuda_device)).cpu().numpy()
    np.testing.assert_array_equal(got, oracle.dot_matrix(x, y)[ri, ci])


@pytest.mark.parametrize("name,n,d,k,csls", [
    ("c1_k10", 10500, 1200, 10, True),
    ("c1_k3", 10500, 1200, 3, True),
    ("c2_k10", 10500, 1800, 10, True),
    ("c3_k10", 10277, 1200, 10, True),
    ("c1_nocsls", 10500, 1200, 10, False),
])
def test_baseline_config_against_the_fp32_oracle(cuda_device, name, n, d, k, csls):
    oracle.set_threads()
    x, y = _clustered(n, d, 8.0, 3408)
    X, Y, xn, yn = _prep(x, y, cuda_device)
    ref = oracle.align_eval(x, y, csls, k)
    res = _run(X, Y, xn, yn, n, k, csls, want_top3=True)[0]
    _assert_equal_to_oracle(res, ref, csls)
    hits1 = float(evaluate.metrics_from_ranks(res.rank_l2r).acc[0])
    assert 0.3 < hits1 < 0.999, hits1
    assert (res.top3_idx.cpu().numpy() == ref["top3"]).all(axis=1).mean() >= 0.999
    print(f"\n[fp32 {name}] deferred {res.info['rank_sweep']['deferred']}, flagged rows/cols "
          f"{res.info['neighbourhoods'].get('rows', {}).get('flagged')}/{res.info['neighbourhoods'].get('cols', {}).get('flagged')}")
    for world in (2, 8):
        _assert_equal_to_oracle(_run(X, Y, xn, yn, n, k, csls, world=world)[world - 1], ref, csls)
    if name == "c1_k10":
        # teeth: on these unrounded rows the bf16 evaluation moves ranks, the fp32 one does not
        Xb, xnb = ops.prep_bf16(torch.from_numpy(x).to(cuda_device), None, normalize=False)
        Yb, ynb = ops.prep_bf16(torch.from_numpy(y).to(cuda_device), None, normalize=False)
        b = evaluate.align_ranks(Xb, Yb, xnb, ynb, n, k, csls)
        moved = int((b.rank_l2r.cpu().numpy() != ref["rank_l2r"]).sum() + (b.rank_r2l.cpu().numpy() != ref["rank_r2l"]).sum())
        print(f"[fp32 {name}] ranks the bf16 evaluation moves: {moved}")
        assert moved >= 1


def test_public_entry_point(cuda_device):
    """evaluate_alignment(precision="fp32") gathers, normalises and evaluates: the oracle on F.normalize's rows."""
    rng = np.random.RandomState(4)
    emb = rng.randn(3000, 300).astype(np.float32)
    emb[1500:] = emb[:1500] + 2.0 * rng.randn(1500, 300).astype(np.float32)
    left, right = np.arange(1500), np.arange(1500, 3000)
    out = evaluate.evaluate_alignment(torch.from_numpy(emb).to(cuda_device), torch.from_numpy(left).to(cuda_device),
                                      torch.from_numpy(right).to(cuda_device), True, 10, want_top3=True, precision="fp32")
    S, _ = fp32.prep(torch.from_numpy(emb).to(cuda_device), None, True, 0)
    fe = S.rows[:, :300].cpu().numpy()                              # the device's F.normalize (bit-equal to prep_bf16's)
    ref = oracle.align_eval(fe[left], fe[right], True, 10)
    _assert_equal_to_oracle(out["ranks"], ref, True)
    assert out["ranks"].info["precision"] == "fp32"


@pytest.mark.parametrize("name", golden_names("eval_"))
def test_bf16_representable_goldens(cuda_device, name):
    """Inputs that are exact in bf16 (m = 0): the fp32 mode equals the bf16 mode bit for bit and the recorded ranks."""
    fx = load_golden(name)
    k, csls = int(fx["k"]), bool(fx["csls"])
    x, y = fx["x"], fx["y"]
    assert np.array_equal(oracle.bf16_round(x), x) and np.array_equal(oracle.bf16_round(y), y)
    n = x.shape[0]
    X, Y, xn, yn = _prep(x, y, cuda_device)
    assert not X.split[:, :X.shape[1]].float().any() and not Y.split[:, X.shape[1]:2 * X.shape[1]].float().any()
    res = _run(X, Y, xn, yn, n, k, csls, want_top3=True)[0]
    Xb, Yb = ops.prep_bf16(torch.from_numpy(x).to(cuda_device), None, False), ops.prep_bf16(torch.from_numpy(y).to(cuda_device), None, False)
    b = evaluate.align_ranks(Xb[0], Yb[0], Xb[1], Yb[1], n, k, csls, want_top3=True)
    for f in ("rank_l2r", "rank_r2l", "g", "top3_idx") + (("nv1", "nv2") if csls else ()):
        assert torch.equal(getattr(res, f), getattr(b, f)), f
    np.testing.assert_array_equal(res.rank_l2r.cpu().numpy(), fx["rank_l2r"])
    np.testing.assert_array_equal(res.rank_r2l.cpu().numpy(), fx["rank_r2l"])
    np.testing.assert_array_equal(res.top3_idx.cpu().numpy(), fx["top3"])
    for side, ranks in (("l2r", res.rank_l2r), ("r2l", res.rank_r2l)):
        m = evaluate.metrics_from_ranks(ranks)
        np.testing.assert_array_equal(m.acc, fx[f"acc_{side}"])
        assert m.mr == float(fx[f"mr_{side}"]) and m.mrr == float(fx[f"mrr_{side}"])


def test_two_sweep_size_against_the_fp32_oracle(cuda_device):
    """n = TWO_SWEEP_MIN_N + 1: the one-pass and the two-sweep paths on split operands, 1 and 4 ranks."""
    oracle.set_threads()
    n, d, k = evaluate.TWO_SWEEP_MIN_N + 1, 384, 10
    x, y = _clustered(n, d, 8.0, 3409)
    X, Y, xn, yn = _prep(x, y, cuda_device)
    ref = oracle.align_eval_stream(x, y, True, k, 2048)
    for one_pass, kernel in ((True, "sim_kernel<EpiOnePass>"), (False, "sim_kernel<EpiRowColTopK>")):
        for _attempt in range(4):
            sweeps = []
            ops.SWEEP_EVENT_SINK = sweeps
            try:
                res = _run(X, Y, xn, yn, n, k, True, one_pass=one_pass)[0]
            finally:
                ops.SWEEP_EVENT_SINK = None
            assert kernel in [nm for nm, *_ in sweeps]
            _assert_equal_to_oracle(res, ref, True)          # exact whatever the one-pass evaluation fell back to
            # the wider fp32 band streams more rank candidates: a first evaluation may overflow the initial per-CTA
            # stream (classic sweep 2, exact) and raise the capacity for the next one
            if not one_pass or res.info["one_pass"]["fallback"] != "rank stream overflow":
                break
        if one_pass:
            info = res.info["one_pass"]
            assert info["fallback"] is None, info
            print(f"\n[fp32 one-pass] n={n}: streamed {info['streamed']}, deferred {info['deferred']}, failed guesses "
                  f"rows/cols {info['failed_rows']}/{info['failed_cols']}")
        _assert_equal_to_oracle(_run(X, Y, xn, yn, n, k, True, world=4, one_pass=one_pass)[1], ref, True)


def _adversarial_rows(n, d, seed):
    """The rows of test_eval_baseline_gpu's band measurement (clustered, all-positive, constant, spiky, sign-alternating,
    near-duplicates, exact duplicates through X = Y), normalised but NOT rounded to bf16."""
    rng = np.random.RandomState(seed)
    q = n // 8
    centres = rng.randn(16, d).astype(np.float32)
    dense = rng.randn(2 * q, d).astype(np.float32) + centres[rng.randint(0, 16, 2 * q)]
    pos = np.abs(rng.randn(q, d)).astype(np.float32)
    const = np.ones((q, d), np.float32) * (1 + 1e-3 * rng.rand(q, 1).astype(np.float32))
    spiky = (rng.randn(q, d) * (rng.rand(q, d) < 0.02)).astype(np.float32) + 1e-3 * rng.randn(q, d).astype(np.float32)
    alt = pos * np.where(np.arange(d) % 2 == 0, 1.0, -1.0).astype(np.float32)
    near = dense[:q] + 1e-3 * rng.randn(q, d).astype(np.float32)
    rest = rng.randn(n - 7 * q, d).astype(np.float32)
    return oracle.normalize_rows(np.concatenate([dense, pos, const, spiky, alt, near, rest], 0))


@pytest.mark.parametrize("d", [1200, 1856])
def test_split_tensor_core_error_on_1e9_pairs(cuda_device, d):
    """E_tc of the split operands: 32 768^2 = 1.07e9 pairs per width through ops.sim_write ([m|h|h] . [h|m|h]), against
    (a) the exact fp64 value of the three products (the tensor core's accumulation error alone, what
    FP32_TC_DOT_ERR_PER_K bounds) and (b) an fp64 GEMM of the fp32 rows (everything: accumulation + split + rounding,
    what fp32.tc_margin must cover with a 4x margin on (a))."""
    n = 32768
    x = torch.from_numpy(_adversarial_rows(n, d, 77)).to(cuda_device)
    A, _ = fp32.prep(x, None, False, 0)
    B, _ = fp32.prep(x, None, False, 1)
    dpad = A.shape[1]
    S = ops.sim_write(A.split, B.split, None, None, n, n, 0)
    Ad, Bd, Xd = A.split.double(), B.split.double(), A.rows.double()
    worst_tc = worst_all = 0.0
    pairs = 0
    for r0 in range(0, n, 2048):
        blk = S[r0:r0 + 2048].double()
        worst_tc = max(worst_tc, float((blk - Ad[r0:r0 + 2048] @ Bd.t()).abs().max()))
        worst_all = max(worst_all, float((blk - Xd[r0:r0 + 2048] @ Xd.t()).abs().max()))
        pairs += blk.numel()
    assert pairs >= 1_000_000_000
    model = fp32.FP32_TC_DOT_ERR_PER_K * dpad
    print(f"\n[split] D={d}: max |s_tc - split_fp64| = {worst_tc:.3e} ({worst_tc / dpad:.2e} per k), max |s_tc - s_fp64| = "
          f"{worst_all:.3e} over {pairs:.3e} pairs; model {model:.3e}, margin {fp32.tc_margin(dpad):.3e}, "
          f"bf16 margin {ops.tc_margin(dpad):.3e}")
    assert worst_tc <= model, worst_tc
    assert worst_all <= model + fp32.SPLIT_REL_ERR + fp32.HALF_ULP, worst_all
    assert 4 * worst_tc + fp32.SPLIT_REL_ERR + fp32.HALF_ULP <= fp32.tc_margin(dpad)
