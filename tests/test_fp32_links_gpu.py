"""GPU: the trainer's link searches on UNROUNDED fp32 rows — mining.mutual_nearest / iter_new_links and
seeds.topk_similarity_entries / visual_pivot_induction with precision="fp32" (snag_b200.fp32 backend) — bit-equal to the
oracle (fp64 index-order dots on the fp32 rows) and to the reference's goldens; on inputs where bf16 rounding moves a
near-tied argmin or top-K entry the bf16 mode differs from the oracle and the fp32 mode does not; on bf16-representable
rows both modes agree; and one patched reference run with --link-precision fp32 through an iterative-learning epoch."""
from __future__ import annotations

import logging
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

from baseline import harness
from oracle import oracle
from snag_b200 import mining, seeds
from tests.conftest import golden_names, load_golden

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _mining_rows(n1, n2, d, sigma, rounded=False):
    """test_mining_vs_oracle's generator (16 cluster centres, noisy permuted copies), normalised, by default NOT rounded."""
    rng = np.random.RandomState(n1 + n2)
    centres = rng.randn(16, d).astype(np.float32)
    x = rng.randn(max(n1, n2), d).astype(np.float32) + centres[rng.randint(0, 16, max(n1, n2))]
    y = x + sigma * rng.randn(max(n1, n2), d).astype(np.float32)
    rnd = oracle.bf16_round if rounded else (lambda a: a)
    x = rnd(oracle.normalize_rows(x))[:n1]
    y = rnd(oracle.normalize_rows(y))[rng.permutation(max(n1, n2))[:n2]]
    return np.ascontiguousarray(x), np.ascontiguousarray(y)


def _seed_rows(n_l, n_r, d, rounded=False):
    """test_topk_entries_vs_oracle's generator (noisy pairs plus a hub), normalised, by default NOT rounded."""
    rng = np.random.RandomState(n_l + n_r)
    base = rng.randn(max(n_l, n_r), d).astype(np.float32)
    x = base[:n_l] + 0.7 * rng.randn(n_l, d).astype(np.float32)
    y = base[:n_r] + 0.7 * rng.randn(n_r, d).astype(np.float32)
    if n_r > 3:
        x[: n_l // 2] += 3.0 * y[2]                      # a hub
    rnd = oracle.bf16_round if rounded else (lambda a: a)
    return rnd(oracle.normalize_rows(x)), rnd(oracle.normalize_rows(y))


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _np(*ts):
    return [t.cpu().numpy() for t in ts]


@pytest.mark.parametrize("n1,n2,d,sigma", [(5000, 4500, 300, 3.0), (20000, 9000, 128, 2.0), (130, 3000, 64, 1.0),
                                           (1, 5, 64, 1.0)])
def test_mining_fp32_vs_oracle(cuda_device, n1, n2, d, sigma):
    x, y = _mining_rows(n1, n2, d, sigma)
    ref = oracle.mutual_nn(x, y)
    out = _np(*mining.mutual_nearest(_t(x, cuda_device), _t(y, cuda_device), precision="fp32"))
    for got, want in zip(out, ref):
        np.testing.assert_array_equal(got, want)
    # iter_new_links on an entity table holding both sides (interleaved ids), refresh and filter epochs
    emb = np.zeros((n1 + n2 + 7, d), np.float32)
    ids = np.random.RandomState(7).permutation(emb.shape[0])
    left, right = ids[:n1].tolist(), ids[n1:n1 + n2].tolist()
    emb[left], emb[right] = x, y
    links = oracle.iter_new_links(left, right, emb, [], True)
    assert mining.iter_new_links(left, right, _t(emb, cuda_device), [], True, precision="fp32") == links
    prev = links[::2] + [(left[0], right[-1])]
    assert (mining.iter_new_links(left, right, _t(emb, cuda_device), prev, False, precision="fp32")
            == oracle.iter_new_links(left, right, emb, prev, False))


@pytest.mark.parametrize("name", golden_names("mining_"))
def test_mining_fp32_golden(cuda_device, name):
    """The reference's own Iter_new_links outputs on its fp32 rows."""
    fx = load_golden(name)
    emb = _t(fx["emb"], cuda_device)
    left, right = fx["left"].tolist(), fx["right"].tolist()
    pl, pr, dl, dr = _np(*mining.mutual_nearest(emb[left], emb[right], precision="fp32"))
    np.testing.assert_array_equal(pl, fx["preds_l"])
    np.testing.assert_array_equal(pr, fx["preds_r"])
    np.testing.assert_allclose(dl, fx["dmin_l"], atol=2e-6, rtol=0)     # the reference's fp32 GEMM, not fp64 dots
    np.testing.assert_allclose(dr, fx["dmin_r"], atol=2e-6, rtol=0)
    ref = oracle.mutual_nn(fx["emb"][left], fx["emb"][right])
    np.testing.assert_array_equal(dl, ref[2])
    np.testing.assert_array_equal(dr, ref[3])
    assert (mining.iter_new_links(left, right, emb, [], True, precision="fp32")
            == [tuple(t) for t in fx["links_refresh"].tolist()])
    prev = [tuple(t) for t in fx["prev"].tolist()]
    assert (mining.iter_new_links(left, right, emb, prev, False, precision="fp32")
            == [tuple(t) for t in fx["links_filter"].tolist()])


@pytest.mark.parametrize("n_l,n_r,d,K", [(2000, 1500, 300, 5000), (700, 5000, 2048, 20000), (50, 40, 64, 2000), (33, 1, 8, 5),
                                         (600, 3000, 4096, 20000)])
def test_topk_entries_fp32_vs_oracle(cuda_device, n_l, n_r, d, K):
    """The grid of test_topk_entries_vs_oracle (hubs, K beyond the 16-per-row pools, a single right column) on unrounded
    rows, plus D = 4096 (FBDB15K's image width: a 12 288-wide split operand)."""
    x, y = _seed_rows(n_l, n_r, d)
    rows, cols, sims = _np(*seeds.topk_similarity_entries(_t(x, cuda_device), _t(y, cuda_device), K, precision="fp32"))
    orow, ocol, osim = oracle.topk_similarity_entries(x, y, K)
    np.testing.assert_array_equal(sims, osim)
    np.testing.assert_array_equal(rows, orow)
    np.testing.assert_array_equal(cols, ocol)


@pytest.mark.parametrize("name", golden_names("seeds_"))
def test_seeds_fp32_golden(cuda_device, name, monkeypatch):
    """visual_pivot_induction with the trainer's switch set reproduces the reference's links."""
    fx = load_golden(name)
    left, right, k = fx["left"].tolist(), fx["right"].tolist(), int(fx["unsup_k"])
    feats = torch.from_numpy(fx["feats"])
    rows, cols, sims = _np(*seeds.topk_similarity_entries(feats[left].to(cuda_device), feats[right].to(cuda_device), 100 * k,
                                                          precision="fp32"))
    np.testing.assert_array_equal(rows, fx["top_rows"])
    np.testing.assert_array_equal(cols, fx["top_cols"])
    np.testing.assert_array_equal(sims, fx["top_sims"])
    monkeypatch.setattr(mining, "LINK_PRECISION", "fp32")
    seen = []
    inner = seeds.topk_similarity_entries
    monkeypatch.setattr(seeds, "topk_similarity_entries", lambda *a, **kw: seen.append(kw["precision"]) or inner(*a, **kw))
    links = seeds.visual_pivot_induction(types.SimpleNamespace(unsup_k=k), left, right, feats,
                                         [tuple(t) for t in fx["ills"].tolist()], logging.getLogger("test_fp32_links"))
    assert seen == ["fp32"]
    np.testing.assert_array_equal(links, fx["links"])


def test_mining_teeth(cuda_device):
    """Two near copies of every left row on the right: which one is nearer is decided below bf16's resolution."""
    rng = np.random.RandomState(11)
    x = oracle.normalize_rows(rng.randn(3000, 256).astype(np.float32))
    y = oracle.normalize_rows(np.concatenate([x + 0.01 * rng.randn(3000, 256).astype(np.float32) for _ in range(2)]))
    ref = oracle.mutual_nn(x, y)
    xt, yt = _t(x, cuda_device), _t(y, cuda_device)
    bf = _np(*mining.mutual_nearest(xt, yt))
    assert (bf[0] != ref[0]).any()
    f32 = _np(*mining.mutual_nearest(xt, yt, precision="fp32"))
    for got, want in zip(f32, ref):
        np.testing.assert_array_equal(got, want)


def test_seeds_teeth(cuda_device):
    """Every left row has one close partner on the right; the top K of those pairs is ordered below bf16's resolution."""
    rng = np.random.RandomState(12)
    x = oracle.normalize_rows(rng.randn(1500, 256).astype(np.float32))
    y = oracle.normalize_rows(x + 0.05 * rng.randn(1500, 256).astype(np.float32))
    K = 1000
    orow, ocol, osim = oracle.topk_similarity_entries(x, y, K)
    xt, yt = _t(x, cuda_device), _t(y, cuda_device)
    brow, bcol, _ = _np(*seeds.topk_similarity_entries(xt, yt, K))
    assert not (np.array_equal(brow, orow) and np.array_equal(bcol, ocol))
    rows, cols, sims = _np(*seeds.topk_similarity_entries(xt, yt, K, precision="fp32"))
    np.testing.assert_array_equal(rows, orow)
    np.testing.assert_array_equal(cols, ocol)
    np.testing.assert_array_equal(sims, osim)


def test_both_modes_agree_on_bf16_representable_rows(cuda_device):
    x, y = _mining_rows(5000, 4500, 300, 3.0, rounded=True)
    xt, yt = _t(x, cuda_device), _t(y, cuda_device)
    for a, b in zip(_np(*mining.mutual_nearest(xt, yt)), _np(*mining.mutual_nearest(xt, yt, precision="fp32"))):
        np.testing.assert_array_equal(a, b)
    x, y = _seed_rows(700, 5000, 2048, rounded=True)
    xt, yt = _t(x, cuda_device), _t(y, cuda_device)
    for a, b in zip(_np(*seeds.topk_similarity_entries(xt, yt, 20000)),
                    _np(*seeds.topk_similarity_entries(xt, yt, 20000, precision="fp32"))):
        np.testing.assert_array_equal(a, b)


_COUNTING_LAUNCHER = """
import sys
from snag_b200 import mining, patch
inner, calls = mining.Iter_new_links, []
def counted(*a, **kw):
    calls.append(mining.LINK_PRECISION)
    return inner(*a, **kw)
mining.Iter_new_links = counted          # installed on the reference class by patch()
try:
    opts = patch.parse_args(sys.argv[1:])
    patch.run_main(opts[1], opts[2], opts[0], opts.link_precision)
finally:
    print("Iter_new_links calls:", calls)
"""


@pytest.mark.skipif(harness.ref_root() is None, reason="no reference checkout (baseline/install_ref.py)")
def test_patched_reference_mines_in_fp32(cuda_device, tmp_path):
    ref = harness.ref_root()
    data = tmp_path / "data"
    harness.write_dataset(str(data), n_side=1500, n_links=1000)
    argv = harness.main_argv(str(data), epochs=6, batch_size=256, extra=["--il", "--il_start", "1"])
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([harness.STUBS, ROOT, env.get("PYTHONPATH", "")])
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    r = subprocess.run([sys.executable, "-c", _COUNTING_LAUNCHER, "--link-precision", "fp32", ref] + argv, cwd=ref, env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("Iter_new_links calls:")]
    assert line and "'fp32'" in line[-1] and "'bf16'" not in line[-1], r.stdout[-4000:]
