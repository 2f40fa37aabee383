"""CPU: the fp64 loss reference and its error bound (tests/loss_fp64_reference.py) are not vacuous. Faults of the shape
kernel bugs take (one row, one diagonal entry, one block of 128 anchors, one padded column, one ragged edge) are
planted in reference data and must be rejected; the reference with the kernels' own roundings must be accepted; and
the bound's rounding terms hold against an independent fp64 evaluation that rounds G to bf16 with the oracle."""
from __future__ import annotations

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import oracle
from snag_b200 import loss as sloss, ops
from tests import loss_fp64_reference as ref64


def _problem(B, D, seed, inv_tau=10.0, ab=0.3):
    g = torch.Generator().manual_seed(seed)
    N = 2 * B + 7
    emb = torch.randn((N, D), generator=g)
    perm = torch.randperm(N, generator=g)
    il, ir = perm[:B].contiguous(), perm[B:2 * B].contiguous()
    emb[ir] = emb[il] + 0.7 * torch.randn((B, D), generator=g)
    z = F.normalize(emb, dim=1)
    a, b = ref64.round_bf16(z[il].double()), ref64.round_bf16(z[ir].double())
    w = torch.rand((B,), generator=g, dtype=torch.float64) + 0.5
    r = ref64.icl_reference(a, b, emb, il, ir, inv_tau, ab, w)
    return dict(emb=emb, il=il, ir=ir, a=a, b=b, w=w, inv_tau=inv_tau, ab=ab, ref=r)


def _report(p, demb, nll_a=None, dz_a=None, name="planted"):
    r = p["ref"]
    rep = ref64.Report(name)
    rep.rows("demb", demb, r["demb"], r["demb_bound"])
    if nll_a is not None:
        rep.elementwise("nll_a", nll_a, r["nll_a"], r["nll_bound_a"])
    if dz_a is not None:
        rep.elementwise("dz_a", dz_a, r["dz_a"], r["dz_bound_a"])
    return rep


def _demb_from(p, dz_a, dz_b):
    e = torch.zeros_like(p["ref"]["demb"])
    e.index_add_(0, p["il"], ref64.normalize_bwd(p["emb"], p["il"], dz_a))
    e.index_add_(0, p["ir"], ref64.normalize_bwd(p["emb"], p["ir"], dz_b))
    return e


def _kernel_like(p):
    """What the recomputing backward computes, in fp64 apart from its roundings: G rounded once to bf16, then G . Y."""
    r, a, b, n = p["ref"], p["a"], p["b"], p["a"].shape[0]
    ca, cb = p["ab"] * p["w"] / n, (1 - p["ab"]) * p["w"] / n
    Ga, _, _ = ref64.icl_dlogits(r["Pa"], r["Pb"], ca, cb, p["inv_tau"])
    Gb, _, _ = ref64.icl_dlogits(r["Pb"], r["Pa"], cb, ca, p["inv_tau"])
    return ref64.round_bf16(Ga) @ torch.cat([b, a], 0), ref64.round_bf16(Gb) @ torch.cat([a, b], 0)


def _frobenius(x, y):
    return float((x - y).norm() / y.norm())


def test_accepts_the_reference_with_bf16_rounded_dlogits():
    p = _problem(300, 64, 1)
    dz_a, dz_b = _kernel_like(p)
    rep = _report(p, _demb_from(p, dz_a, dz_b), p["ref"]["nll_a"].float(), dz_a, "bf16 G")
    rep.check()
    assert rep.ratios["demb"] > 1e-3          # the bound is not orders of magnitude above the rounding it describes


def test_rejects_one_row_scaled_that_the_frobenius_criterion_accepts():
    p = _problem(300, 64, 2)
    demb = p["ref"]["demb"].clone()
    row = int(p["il"][137])
    demb[row] *= 1 + 2.0 ** -4
    assert _frobenius(demb, p["ref"]["demb"]) < 1e-2          # test_loss_gpu.py's aggregate check passes this fault
    assert _report(p, demb).worst() > 1.0


def test_rejects_a_dropped_cross_diagonal_term():
    p = _problem(300, 64, 3)
    bad = ref64.icl_reference(p["a"], p["b"], p["emb"], p["il"], p["ir"], p["inv_tau"], p["ab"], p["w"],
                              fault={"drop_diag": 41})
    rep = _report(p, bad["demb"], dz_a=bad["dz_a"])
    assert rep.ratios["demb"] > 1.0 and rep.ratios["dz_a"] > 1.0


def test_rejects_a_zeroed_block_of_one_ranks_share():
    B, world = 600, 2
    p = _problem(B, 64, 4)
    r0, r1, per = sloss.AnchorShard(world=world, rank=1).bounds(B)
    assert (r0, r1) == (384, 600)
    dz_a = p["ref"]["dz_a"].clone()
    dz_a[r0:r0 + 128] = 0.0                                    # the rank's first block of 128 anchors lost
    rep = _report(p, _demb_from(p, dz_a, p["ref"]["dz_b"]), dz_a=dz_a)
    assert rep.ratios["demb"] > 1.0 and rep.ratios["dz_a"] > 1.0


def test_rejects_a_padded_column_leak():
    """dz as the kernels return it, [B, Dpad]: the bound of a padded column is 0, so any value there is rejected."""
    B, D = 200, 63
    p = _problem(B, D, 5)
    dpad = ops.round_up(D, 64)
    pad = lambda t: F.pad(t, (0, dpad - D))
    got = pad(p["ref"]["dz_a"]).clone()
    got[17, D] = 1e-6 * float(p["ref"]["dz_a"].abs().max())
    rep = ref64.Report("pad")
    rep.elementwise("dz_a", got, pad(p["ref"]["dz_a"]), pad(p["ref"]["dz_bound_a"]))
    assert rep.worst() > 1.0
    clean = ref64.Report("pad")
    clean.elementwise("dz_a", pad(p["ref"]["dz_a"]).float(), pad(p["ref"]["dz_a"]), pad(p["ref"]["dz_bound_a"]))
    clean.check()


def test_rejects_the_last_anchor_of_a_ragged_batch_dropped_from_the_column_terms():
    B = 257
    p = _problem(B, 96, 6)
    bad = ref64.icl_reference(p["a"], p["b"], p["emb"], p["il"], p["ir"], p["inv_tau"], p["ab"], p["w"],
                              fault={"drop_col": B - 1})
    assert _report(p, bad["demb"]).worst() > 1.0


def test_rejects_a_wrong_nll():
    p = _problem(129, 64, 7)
    nll = p["ref"]["nll_a"].clone()
    nll[128] += 1e-3                                           # one anchor of the ragged last block
    assert _report(p, p["ref"]["demb"], nll).ratios["nll_a"] > 1.0


@pytest.mark.parametrize("inv_tau", [2.0, 10.0, 20.0])
def test_rounding_terms_hold_against_an_independent_bf16_evaluation(inv_tau):
    """The ubf |G| |Y| term (one bf16 rounding of G), the saved-E form (E rounded, then G) and IAL's centred
    difference, against fp64 products of G rounded with oracle.bf16_round (numpy, independent of torch's rounding)."""
    p = _problem(256, 64, 8, inv_tau)
    r, a, b, n = p["ref"], p["a"], p["b"], 256
    Y = torch.cat([b, a], 0)
    ca, cb = p["ab"] * p["w"] / n, (1 - p["ab"]) * p["w"] / n
    G, Gabs, dg = ref64.icl_dlogits(r["Pa"], r["Pb"], ca, cb, inv_tau)
    rnd = lambda t: torch.from_numpy(oracle.bf16_round(t.numpy().astype(np.float32)).astype(np.float64))
    Ya = Y.abs()
    err = (rnd(G) @ Y - G @ Y).abs()
    term = ref64.UBF * G.abs() @ Ya
    ratio = float((err / term).max())
    assert 0.05 < ratio <= 1.0, ratio
    # saved E: E rounded to bf16, then the coefficients applied and G rounded again
    E = torch.exp((torch.cat([a @ b.t(), (a @ a.t()).fill_diagonal_(-np.inf)], 1) - 1.0) * inv_tau)
    cr = ca * torch.exp(inv_tau - r["lse_a"])
    cc = cb * torch.exp(inv_tau - r["lse_b"])
    coef = torch.cat([cr[:, None] + cc[None, :], cr[:, None] + cr[None, :]], 1) * inv_tau
    assert float(((coef * E - Gabs).abs() / Gabs.clamp_min(1e-300)).max()) < 1e-12    # the kernels' form of G
    Gs = coef * rnd(E)
    Gs[torch.arange(n), torch.arange(n)] -= dg
    err2 = (rnd(Gs) @ Y - G @ Y).abs()
    term2 = (ref64.UBF * G.abs() + ref64.UBF * Gabs) @ Ya
    assert float((err2 / term2).max()) <= 1.0
    # IAL: the two centred matrices and their difference rounded
    ebar = float(np.exp(-inv_tau))
    Gs_c, Gt_c = coef * (E - ebar), 0.9 * coef * (E - ebar).flip(1)
    Gs_c[:, n:].fill_diagonal_(0.0)
    Gt_c[:, n:].fill_diagonal_(0.0)
    err3 = (rnd(rnd(Gs_c) - rnd(Gt_c)) @ Y - (Gs_c - Gt_c) @ Y).abs()
    term3 = ref64.UBF * (Gs_c.abs() + Gt_c.abs() + (Gs_c - Gt_c).abs()) @ Ya
    assert float((err3 / term3).max()) <= 1.0


def test_reference_matches_autograd_of_the_reference_op_sequence():
    """The closed-form fp64 gradients against torch autograd of model/SNAG_loss.py's op sequence, in fp64."""
    p = _problem(130, 48, 9, 10.0, 0.4)
    B = 130
    e = p["emb"].double().requires_grad_(True)
    z = F.normalize(e, dim=1)
    z = z + (torch.zeros_like(z).index_copy(0, p["il"], p["a"]).index_copy(0, p["ir"], p["b"]) - z).detach()
    za, zb = z[p["il"]], z[p["ir"]]
    eye = torch.eye(B, dtype=torch.float64) * 1e9
    la = torch.cat([za @ zb.t(), za @ za.t() - eye], 1) * 10.0
    lb = torch.cat([zb @ za.t(), zb @ zb.t() - eye], 1) * 10.0
    ar = torch.arange(B)
    nll_a, nll_b = -F.log_softmax(la, 1)[ar, ar], -F.log_softmax(lb, 1)[ar, ar]
    loss = 0.4 * (nll_a * p["w"]).sum() / B + 0.6 * (nll_b * p["w"]).sum() / B
    loss.backward()
    r = p["ref"]
    assert abs(loss.item() - float(r["loss"])) < 1e-12
    assert float((nll_a - r["nll_a"]).abs().max()) < 1e-12
    assert float((e.grad - r["demb"]).abs().max()) < 1e-12 * float(r["demb"].abs().max())


def test_ial_reference_matches_autograd():
    B, Ds, Dt, inv_tau = 120, 40, 72, 2.0
    g = torch.Generator().manual_seed(10)
    N = 2 * B + 5
    src, tar = torch.randn((N, Ds), generator=g), torch.randn((N, Dt), generator=g)
    perm = torch.randperm(N, generator=g)
    il, ir = perm[:B].contiguous(), perm[B:2 * B].contiguous()
    zs, zt = ref64.round_bf16(F.normalize(src, dim=1).double()), ref64.round_bf16(F.normalize(tar, dim=1).double())
    r = ref64.ial_reference(zs[il], zs[ir], zt[il], zt[ir], src, il, ir, inv_tau, 0.3, 0.1, "mean")
    e = src.double().requires_grad_(True)
    z = F.normalize(e, dim=1)
    z = z + (zs - z).detach()
    eye = torch.eye(B, dtype=torch.float64) * 1e9
    out = 0
    for l, rr, wgt in ((il, ir, 0.3), (ir, il, 0.7)):
        pl = torch.cat([z[l] @ z[rr].t(), z[l] @ z[l].t() - eye], 1) * inv_tau
        ql = torch.cat([zt[l] @ zt[rr].t(), zt[l] @ zt[l].t() - eye], 1) * inv_tau
        out = out + wgt * F.kl_div(F.log_softmax(pl, 1), F.softmax(ql, 1), reduction="none").mean()
    out = 0.1 * out
    out.backward()
    assert abs(float(out) - r["loss"]) < 1e-12 * max(1.0, abs(float(out))) + 1e-15
    assert float((e.grad - r["demb"]).abs().max()) < 1e-10 * float(r["demb"].abs().max())
    assert r["loss_bound"] > 0 and float(r["demb_bound"].max()) > 0


@pytest.mark.parametrize("tau", [0.02, 1.0 / 41])
def test_temperatures_beyond_the_ftz_safe_range_are_refused(tau):
    """exp((s - 1)/tau) is evaluated as ex2.approx.ftz: below 2^-126 it flushes to 0, and a row whose every similarity
    is negative enough would sum to 0 beyond 1/tau = 43.3 (s >= -(1 + 2^-8)^2 for bf16-rounded unit rows), and the
    backward's row scale exp(1/tau - lse) / tau must stay finite in fp32."""
    emb = torch.randn(40, 16)
    links = np.stack([np.arange(10), np.arange(20, 30)], 1)
    with pytest.raises(ValueError, match="1/tau"):
        sloss.icl_loss(tau=tau)(emb, links)
    with pytest.raises(ValueError, match="1/tau"):
        sloss.ial_loss(tau=tau, ab_weight=0.5, zoom=0.1)(emb, emb, links)
    span = 2 * (1 + 2.0 ** -8) ** 2 * sloss.MAX_INV_TAU
    assert span * np.log2(np.e) <= 126 and np.exp(span) * sloss.MAX_INV_TAU < 2.0 ** 128


def test_norm_false_refuses_an_effective_temperature_beyond_the_range():
    """norm=False folds 4^e into 1/tau: 1/tau = 2 with rows of norm ~ 6 (e = 3) is 128 in the kernels"""
    emb = torch.randn(40, 16) * 1.5
    links = np.stack([np.arange(10), np.arange(20, 30)], 1)
    with pytest.raises(ValueError, match="norm=False"):
        sloss.icl_loss(tau=0.5)(emb, links, norm=False)
