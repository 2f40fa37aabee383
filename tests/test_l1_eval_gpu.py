"""GPU: the fused --distance 1 evaluation (snag_b200.l1 under evaluate._align_ranks_steps) against the reference's
materialised composition and the oracle — ranks, neighbourhood means, ground-truth distances and prediction ids bit
for bit, including exact ties, a filled deferral band, its overflow retry, sharding and sizes the matrix cannot hold."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from oracle import oracle
from snag_b200 import evaluate, l1, ops
from snag_b200._lib import KT
from tests import l1_reference
from tests.conftest import golden_names, load_golden

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


def _steps(X, Y, xn, yn, n, k, csls, top3, world=1):
    res = evaluate.simulate_sharded(
        lambda r: evaluate._align_ranks_steps(l1, X, Y, xn, yn, n, k, csls, top3, world, r, two_sweep=False), world)
    return res[0]


def _operands(x, y, dev):
    X, xn = l1.prep(torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(dev), torch.arange(x.shape[0], device=dev))
    Y, yn = l1.prep(torch.from_numpy(np.ascontiguousarray(y, np.float32)).to(dev), torch.arange(y.shape[0], device=dev))
    return X, Y, xn, yn


def _materialised(fe, left, right, csls, k):
    """The reference's composition on the device: cdist, csls_sim on 1 - distance, ranks of the diagonal."""
    dist = ops.l1_distance(fe.index_select(0, left).contiguous(), fe.index_select(0, right).contiguous())
    nv1 = nv2 = None
    if csls:
        out, nv1, nv2 = ops.csls_sim_matrix(1 - dist, k)
        dist = 1 - out
    r, c = ops.matrix_rank(dist)
    return r, c, nv1, nv2, torch.diagonal(dist).clone()


@pytest.mark.parametrize("name", golden_names("l1_"))
def test_goldens_through_the_fused_route(cuda_device, name):
    fx = load_golden(name)
    n = fx["x"].shape[0]
    emb = torch.from_numpy(np.concatenate([fx["x"], fx["y"]], 0)).to(cuda_device)
    out = evaluate.evaluate_alignment_l1(emb, torch.arange(0, n, device=cuda_device), torch.arange(n, 2 * n, device=cuda_device),
                                         csls=bool(fx["csls"]), csls_k=int(fx["k"]), want_top3=True)
    res = out["ranks"]
    assert not res.info.get("materialised")
    np.testing.assert_array_equal(res.rank_l2r.cpu().numpy(), fx["rank_l2r"])
    np.testing.assert_array_equal(res.rank_r2l.cpu().numpy(), fx["rank_r2l"])
    np.testing.assert_array_equal(res.top3_idx.cpu().numpy(), fx["top3"])


@pytest.mark.parametrize("n", [1500, 10500])
@pytest.mark.parametrize("csls,k", [(True, 3), (True, 10), (False, 10)])
def test_fused_equals_materialised_at_c1_width(cuda_device, n, csls, k):
    rng = np.random.RandomState(n + k)
    d = 1200
    x = rng.randn(n, d).astype(np.float32)
    y = (x + 0.4 * rng.randn(n, d)).astype(np.float32)
    emb = torch.from_numpy(np.concatenate([x, y], 0)).to(cuda_device)
    left, right = torch.arange(0, n, device=cuda_device), torch.arange(n, 2 * n, device=cuda_device)
    out = evaluate.evaluate_alignment_l1(emb, left, right, csls=csls, csls_k=k)
    r, c, nv1, nv2, g = _materialised(torch.nn.functional.normalize(emb), left, right, csls, k)
    res = out["ranks"]
    assert torch.equal(res.rank_l2r, r) and torch.equal(res.rank_r2l, c)
    assert torch.equal(res.g, g)
    if csls:
        assert torch.equal(res.nv1, nv1) and torch.equal(res.nv2, nv2)


def test_exact_ties_take_the_stable_tie_break(cuda_device):
    rng = np.random.RandomState(5)
    n, d = 700, 40
    x = (rng.randint(-3, 4, (n, d)) / 64.0).astype(np.float32)        # multiples of 2^-6: every sum is exact
    y = x.copy()
    y[::3] = x[(np.arange(0, n, 3) + 1) % n]                           # duplicated rows: tied distances everywhere
    y[1::5] += np.float32(1 / 64)
    X, Y, xn, yn = _operands(x, y, cuda_device)
    for csls, k in ((True, 4), (False, 1)):
        res = _steps(X, Y, xn, yn, n, k, csls, True)
        ref = oracle.align_eval_l1(x, y, csls, k)
        assert (ref["dist"] == ref["g"][:, None]).sum() > 2 * n        # exact ties of the ground truth exist
        np.testing.assert_array_equal(res.rank_l2r.cpu().numpy(), ref["rank_l2r"])
        np.testing.assert_array_equal(res.rank_r2l.cpu().numpy(), ref["rank_r2l"])
        np.testing.assert_array_equal(res.top3_idx.cpu().numpy(), ref["top3"])
        np.testing.assert_array_equal(res.g.cpu().numpy(), ref["g"])


def _near_ties(n, d, seed):
    rng = np.random.RandomState(seed)
    base = oracle.normalize_rows(rng.randn(8, d).astype(np.float32))
    c = rng.randint(0, 8, n)
    x = base[c] + (1e-6 * rng.randn(n, d)).astype(np.float32)          # pairs as close as the rest of their cluster
    y = base[c] + (1e-6 * rng.randn(n, d)).astype(np.float32)
    return oracle.normalize_rows(x), oracle.normalize_rows(y)


def test_near_ties_fill_the_band(cuda_device):
    n, d = 2000, 256
    x, y = _near_ties(n, d, 7)
    X, Y, xn, yn = _operands(x, y, cuda_device)
    res = _steps(X, Y, xn, yn, n, 10, True, True)
    assert l1.LAST_RANK_INFO["deferred"] > n
    ref = oracle.align_eval_l1(x, y, True, 10)
    np.testing.assert_array_equal(res.rank_l2r.cpu().numpy(), ref["rank_l2r"])
    np.testing.assert_array_equal(res.rank_r2l.cpu().numpy(), ref["rank_r2l"])
    np.testing.assert_array_equal(res.nv1.cpu().numpy(), ref["nv1"])
    np.testing.assert_array_equal(res.nv2.cpu().numpy(), ref["nv2"])
    np.testing.assert_array_equal(res.top3_idx.cpu().numpy(), ref["top3"])


def test_band_overflow_is_retried(cuda_device, monkeypatch):
    n, d = 1200, 128
    x, y = _near_ties(n, d, 8)
    X, Y, xn, yn = _operands(x, y, cuda_device)
    monkeypatch.setattr(l1, "BAND_MIN_CAP", 1024)
    monkeypatch.setattr(l1, "BAND_PER_ROW", 0)
    res = _steps(X, Y, xn, yn, n, 5, True, False)
    assert l1.LAST_RANK_INFO["cap"] > 1024                             # the first list overflowed
    ref = oracle.align_eval_l1(x, y, True, 5)
    np.testing.assert_array_equal(res.rank_l2r.cpu().numpy(), ref["rank_l2r"])
    np.testing.assert_array_equal(res.rank_r2l.cpu().numpy(), ref["rank_r2l"])


def test_sweep_error_stays_within_half_the_bound(cuda_device):
    """>= 10^7 adversarial pairs: n2 <= KT targets, so every pair comes back as a candidate of eval_rowtopk."""
    d, n2 = 1200, KT
    rng = np.random.RandomState(11)
    gen = torch.Generator(device=cuda_device).manual_seed(11)
    n1 = 655360
    X = torch.rand((n1, d), device=cuda_device, generator=gen)                       # all positive: worst accumulation
    X[n1 // 4: n1 // 2] = torch.rand((n1 // 4, d), device=cuda_device, generator=gen) * 1e-3
    wide = torch.exp2(torch.randint(-40, 4, (n1 // 4, d), device=cuda_device, generator=gen).float())
    X[n1 // 2: 3 * n1 // 4] = wide * torch.rand((n1 // 4, d), device=cuda_device, generator=gen)  # wide dynamic range
    X[3 * n1 // 4:] = torch.randn((n1 - 3 * n1 // 4, d), device=cuda_device, generator=gen)
    X = torch.nn.functional.normalize(X)
    y = np.abs(rng.randn(n2, d)).astype(np.float32)
    y[n2 // 2:] = -y[n2 // 2:]
    y[0] = 0.0                                                                     # distance = ||x||_1
    Y = torch.nn.functional.normalize(torch.from_numpy(y).to(cuda_device))
    ax, xn = l1.prep(X, torch.arange(n1, device=cuda_device))
    ay, yn = l1.prep(Y, torch.arange(n2, device=cuda_device))
    part, pidx = l1.eval_rowtopk(ax, ay, xn, yn, n1, n2, want_idx=True)
    assert part.shape[0] == 1 and bool((pidx[0] >= 0).all())
    dcan = ops.l1_distance(X.contiguous(), Y.contiguous())                         # canonical: fp64 index order
    cid = pidx[0].long()
    c_can = 1.0 - torch.gather(dcan, 1, cid)
    err = (part[0] - c_can).abs().double()
    S = (xn[:, None] + yn[cid]).double()
    nc = (ax.shape[1] + 31) // 32
    eps = (nc + 18) * 1.01 * U * S
    slack = 2 * U * (1.0 + S)                                                      # the two roundings of 1 - d
    worst = float((err / (eps / 2 + slack)).max())
    assert n1 * n2 >= 10 ** 7
    assert worst <= 1.0, worst


def test_sharded_65537_is_bit_identical(cuda_device):
    n, d = 65537, 300
    rng = np.random.RandomState(21)
    x = oracle.normalize_rows(rng.randn(n, d).astype(np.float32))
    y = oracle.normalize_rows((x + 0.5 * rng.randn(n, d)).astype(np.float32))
    X, Y, xn, yn = _operands(x, y, cuda_device)
    base = _steps(X, Y, xn, yn, n, 10, True, True)
    for world in (2, 4):
        res = _steps(X, Y, xn, yn, n, 10, True, True, world)
        for f in ("rank_l2r", "rank_r2l", "nv1", "nv2", "g", "top3_idx"):
            assert torch.equal(getattr(res, f), getattr(base, f)), (world, f)
    sel = np.sort(rng.choice(n, 16, replace=False))
    a = l1_reference.audit_l1(x[sel], y, sel, True, 10, base.nv2.cpu().numpy(), False)
    np.testing.assert_array_equal(base.rank_l2r.cpu().numpy()[sel], a["rank"])
    np.testing.assert_array_equal(base.nv1.cpu().numpy()[sel], a["nv"])


def test_beyond_the_materialised_size(cuda_device):
    """131 072 pairs: the [n, n] route would need 3 x 69 GB; the fused one runs, 64 sources and 64 targets audited."""
    n, d = 131072, 256
    gen = torch.Generator(device=cuda_device).manual_seed(5)
    x = torch.randn((n, d), device=cuda_device, generator=gen)
    emb = torch.cat([x, x + 0.6 * torch.randn((n, d), device=cuda_device, generator=gen)], 0)
    out = evaluate.evaluate_alignment_l1(emb, torch.arange(0, n, device=cuda_device), torch.arange(n, 2 * n, device=cuda_device),
                                         csls=True, csls_k=10)
    res = out["ranks"]
    fe = torch.nn.functional.normalize(emb).cpu().numpy()
    xs, ys = fe[:n], fe[n:]
    rng = np.random.RandomState(0)
    src = np.sort(rng.choice(n, 64, replace=False))
    tgt = np.sort(rng.choice(n, 64, replace=False))
    a = l1_reference.audit_l1(xs[src], ys, src, True, 10, res.nv2.cpu().numpy(), False)
    np.testing.assert_array_equal(res.rank_l2r.cpu().numpy()[src], a["rank"])
    np.testing.assert_array_equal(res.nv1.cpu().numpy()[src], a["nv"])
    np.testing.assert_array_equal(res.g.cpu().numpy()[src], a["g"])
    b = l1_reference.audit_l1(ys[tgt], xs, tgt, True, 10, res.nv1.cpu().numpy(), True)
    np.testing.assert_array_equal(res.rank_r2l.cpu().numpy()[tgt], b["rank"])
    np.testing.assert_array_equal(res.nv2.cpu().numpy()[tgt], b["nv"])
