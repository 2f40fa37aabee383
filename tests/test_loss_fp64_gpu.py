"""GPU: every forward and backward route of icl_loss / ial_loss against the fp64 reference of
tests/loss_fp64_reference.py, anchor by anchor (lse, NLL) and row by row (d emb, d weight_norm), each against its own
error bound. The operands of the reference are the stacked bf16 rows the kernels consume (ops.icl_stack_prep).
Every test prints the largest error-to-bound ratio per quantity (run with -s to see them)."""
from __future__ import annotations

import math

import numpy as np
import pytest
import torch

from snag_b200 import loss as sloss, ops
from tests import loss_fp64_reference as ref64

pytestmark = pytest.mark.gpu


class _LockstepShard(sloss.AnchorShard):
    """One GPU standing in for `world` ranks that run one after the other. all_gather / all_reduce return the blocks the
    ranks contributed so far (zeros for the missing ones). A rank's forward block depends on its own work only, but its
    backward block (grads="gather") depends on the forward sums of all ranks: a block is complete once every rank has
    run once before it, so the ranks run three times and the last pass (`final`) accepts only blocks of earlier
    complete passes or of this one."""

    def __init__(self, world, rank, store, grads, pass_no, final=False):
        super().__init__(None, grads, None, world, rank)
        self.store, self.pass_no, self.final = store, pass_no, final

    def _blocks(self, t, kind):
        key = (len(self.store.setdefault(("n", self.rank), [])), tuple(t.shape), kind)
        self.store[("n", self.rank)].append(key)
        blocks = self.store.setdefault(key, {})
        blocks[self.rank] = (self.pass_no, t.clone())
        if self.final:
            assert sorted(blocks) == list(range(self.world)), f"{kind}: blocks of ranks {sorted(blocks)} only"
            assert all(p >= self.pass_no - 1 >= 1 for p, _ in blocks.values()), f"{kind}: a block of an incomplete pass"
        return {r: v for r, (_, v) in blocks.items()}

    def all_gather(self, t):
        blocks = self._blocks(t, "gather")
        return torch.stack([blocks.get(r, torch.zeros_like(t)) for r in range(self.world)], 0)

    def all_reduce(self, t):
        blocks = self._blocks(t, "sum")
        return sum(blocks[r] for r in sorted(blocks))


class _Spy:
    """Stands in for loss._IclMany and keeps what the forward returned (per-anchor NLL; lse from the autograd node)."""

    def __init__(self):
        self.calls = []

    def apply(self, *args):
        out = _IclMany.apply(*args)
        self.calls.append((out.detach().clone(), out.grad_fn.saved_tensors[2].clone()))
        return out


_IclMany = sloss._IclMany


def _batch(N, D, B, seed, device, stress=True, anti=False):
    """fp32 table [N, D] and links: correlated pairs plus (stress) a near-duplicate pair, a constant and a duplicated row,
    an entity linked on both sides and a repeated id in idx_l; (anti) anchor 0 anti-correlated with every other row."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    emb = torch.randn((N, D), generator=g, device=device)
    perm = torch.randperm(N, generator=g, device=device)
    il, ir = perm[:B].clone(), perm[B:2 * B].clone()
    emb[ir] = emb[il] + 0.7 * torch.randn((B, D), generator=g, device=device)
    if anti:
        c = torch.randn((1, D), generator=g, device=device)
        emb[:] = 3 * c + 0.3 * torch.randn((N, D), generator=g, device=device)
        emb[il[0]] = -c[0]
    elif stress and B >= 12:
        emb[ir[0]] = emb[il[0]] + 1e-3 * torch.randn((D,), generator=g, device=device)   # P_ii ~ 1
        emb[il[1]] = 1.0
        emb[ir[1]] = 1.0                                                                      # constant rows, tied
        emb[il[3]] = emb[il[2]]                                                               # duplicated row
        ir[5] = il[7]                                                                         # linked on both sides
        il[9] = il[8]                                                                         # repeated id in idx_l
    return emb.contiguous(), il.contiguous(), ir.contiguous()


def _operands(emb, il, ir, normalize=True):
    B = il.numel()
    Bp = ops.round_up(B, 256)
    S3 = ops.icl_stack_prep([emb], il, ir, Bp, normalize)[0]
    D = emb.shape[1]
    return S3[:B, :D].double(), S3[Bp:Bp + B, :D].double()


def _icl_case(route, embs, il, ir, tau, ab, wns, run, saved_e=None, norm=True):
    """run(embs, wns) -> (losses, nll [n, 2, B], lse [n, 2, B], d embs, d wns); checks every table against the reference"""
    inv_tau = 1.0 / tau
    scale = 1.0
    if not norm:                                   # the power-of-two scaling of icl_loss.forward_many
        m2 = max(float(torch.maximum(e[il].square().sum(1).max(), e[ir].square().sum(1).max())) for e in embs)
        e2 = max(0, int(np.ceil(0.5 * np.log2(max(m2, 1e-30)))))
        inv_tau, scale = inv_tau * 4.0 ** e2, 2.0 ** -e2
    losses, nll, lse, gembs, gwns = run(embs, wns)
    rep = ref64.Report(route)
    N = embs[0].shape[0]
    for p, emb in enumerate(embs):
        a, b = _operands(emb * scale if not norm else emb, il, ir, norm)
        w = None
        if wns[p] is not None:
            wl, wr = wns[p][il].double(), wns[p][ir].double()
            w = torch.minimum(wl, wr)
        wide = ops.round_up(emb.shape[1], 64) > ops.FUSED_BWD_MAX_DPAD
        se = saved_e if saved_e is not None else (wide and sloss.SAVE_E and sloss.SYM_FORWARD)
        r = ref64.icl_reference(a, b, emb, il, ir, inv_tau, ab, w, norm=norm, scale=scale, saved_e=se)
        for s, k in (("a", 0), ("b", 1)):
            rep.elementwise("lse", lse[p, k], r[f"lse_{s}"], r[f"lse_bound_{s}"])
            rep.elementwise("nll", nll[p, k], r[f"nll_{s}"], r[f"nll_bound_{s}"])
        rep.elementwise("loss", losses[p].reshape(1), r["loss"].reshape(1), r["loss_bound"])
        rep.rows("demb", gembs[p], r["demb"], r["demb_bound"])
        if wns[p] is not None:
            gw, gwb = ref64.dw_table(r, wl, wr, il, ir, N)
            rep.elementwise("dw", gwns[p], gw, gwb)
        del r
    print(rep)
    return rep.check()


def _public(tau, ab, il, ir, shard=None):
    """forward_many + backward through the public module, with the NLL / lse the forward produced"""

    def run(embs, wns):
        spy = _Spy()
        saved = sloss._IclMany
        sloss._IclMany = spy
        try:
            crit = sloss.icl_loss(tau=tau, ab_weight=ab)
            crit.shard = shard
            e = [t.clone().requires_grad_(True) for t in embs]
            w = [None if t is None else t.clone().requires_grad_(True) for t in wns]
            links = torch.stack([il, ir], 1)
            losses = crit.forward_many(e, links, w, norm=run.norm)
            sum(losses).backward()
        finally:
            sloss._IclMany = saved
        nll, lse = spy.calls[-1]
        return ([x.detach() for x in losses], nll, lse, [t.grad for t in e],
                [None if t is None else t.grad for t in w])

    run.norm = True
    return run


# (route, B, D, tau): a covering grid of batch sizes around the 128 / 256 tile edges, widths around the 64-column
# padding and the 320 / 321 boundary between the fused and the wide backward
ROUTES = [
    ("fused", 1, 8, 0.1), ("fused", 2, 63, 0.1), ("fused", 127, 64, 0.05), ("fused", 129, 65, 0.1),
    ("fused", 256, 300, 0.1), ("fused", 3500, 320, 0.1),
    ("two_kernel", 128, 300, 0.1), ("two_kernel", 255, 65, 0.5), ("two_kernel", 257, 320, 0.1),
    ("wide_saved_e", 127, 321, 0.1), ("wide_saved_e", 257, 1200, 0.1), ("wide_saved_e", 3500, 1800, 0.1),
    ("wide_recompute", 256, 321, 0.1), ("wide_recompute", 1000, 1200, 0.05),
    ("per_side", 129, 64, 0.1), ("per_side", 257, 1200, 0.1), ("per_side", 3500, 300, 0.1),
]


@pytest.mark.parametrize("route,B,D,tau", ROUTES)
def test_icl_route_against_fp64(cuda_device, monkeypatch, route, B, D, tau):
    monkeypatch.setattr(sloss, "FUSED_BACKWARD", route != "two_kernel")
    monkeypatch.setattr(sloss, "SAVE_E", route != "wide_recompute")
    monkeypatch.setattr(sloss, "SYM_FORWARD", route != "per_side")
    emb, il, ir = _batch(2 * B + 31, D, B, B * 7 + D, cuda_device)
    g = torch.Generator(device="cuda").manual_seed(B)
    wn = torch.rand((emb.shape[0],), generator=g, device=cuda_device) + 0.5
    _icl_case(route, [emb], il, ir, tau, 0.3, [wn], _public(tau, 0.3, il, ir))


def test_icl_c5_train_shape_against_fp64(cuda_device):
    """B = 16 384 at D = 1 800, the joint-embedding table of bench.py's c5_train step (wide, saved E)"""
    B, D = 16384, 1800
    emb, il, ir = _batch(2 * B + 100, D, B, 5, cuda_device)
    _icl_case("c5_train", [emb], il, ir, 0.1, 0.5, [None], _public(0.1, 0.5, il, ir))


def _sharded(tau, ab, il, ir, world, grads):
    def run(embs, wns):
        store = {}
        for pass_no in range(3):
            outs = []
            for r in range(world):
                store.pop(("n", r), None)
                shard = _LockstepShard(world, r, store, grads, pass_no, final=pass_no == 2)
                outs.append(_public(tau, ab, il, ir, shard)(embs, wns))
        for o in outs[1:]:                            # every rank holds the same loss and per-anchor statistics
            assert all(torch.equal(x, y) for x, y in zip(o[0], outs[0][0]))
            assert torch.equal(o[1], outs[0][1]) and torch.equal(o[2], outs[0][2])
        if grads == "local":                          # each rank returns its own anchors' rows: the sum is the gradient
            gembs = [sum(o[3][p] for o in outs) for p in range(len(embs))]
        else:                                         # every rank returns the whole gradient: check each one
            for o in outs[1:]:
                for x, y in zip(o[3], outs[0][3]):
                    assert torch.equal(x, y)
            gembs = outs[0][3]
        return outs[0][0], outs[0][1], outs[0][2], gembs, outs[0][4]

    return run


@pytest.mark.parametrize("B,D,world,grads", [
    (1000, 300, 2, "local"), (1000, 300, 2, "gather"), (257, 64, 3, "gather"), (257, 1200, 3, "local"),
    (1000, 1200, 2, "gather"), (300, 96, 8, "local"), (300, 1800, 8, "gather"), (3500, 320, 8, "gather"),
    (2049, 1200, 8, "local")])
def test_icl_sharded_against_fp64(cuda_device, B, D, world, grads):
    """Anchor-sharded loss on `world` lockstep ranks, narrow (fused backward) and wide (two-kernel backward) tables.
    B = 300 at world 8: ranks 3..7 own no anchors; B = 257 at world 3: the last rank owns one anchor."""
    emb, il, ir = _batch(2 * B + 31, D, B, B + D + world, cuda_device)
    g = torch.Generator(device="cuda").manual_seed(world)
    wn = torch.rand((emb.shape[0],), generator=g, device=cuda_device) + 0.5
    _icl_case(f"sharded {grads} w{world}", [emb], il, ir, 0.1, 0.4, [wn], _sharded(0.1, 0.4, il, ir, world, grads),
              saved_e=False)


def test_icl_forward_many_chunks_and_the_width_boundary(cuda_device):
    """18 tables of one width (both 16-table chunk loops, forward and fused backward) and D = 320 with D = 321 in the
    same call (fused and wide backward side by side)."""
    B, N = 300, 700
    widths = [64] * 18 + [320, 321]
    embs, wns = [], []
    _, il, ir = _batch(N, 8, B, 11, cuda_device)
    g = torch.Generator(device="cuda").manual_seed(12)
    for p, d in enumerate(widths):
        e = torch.randn((N, d), generator=g, device=cuda_device)
        e[ir] = e[il] + (0.3 + 0.05 * p) * torch.randn((B, d), generator=g, device=cuda_device)
        embs.append(e)
        wns.append(torch.rand((N,), generator=g, device=cuda_device) + 0.5 if p % 3 == 0 else None)
    _icl_case("forward_many", embs, il, ir, 0.1, 0.5, wns, _public(0.1, 0.5, il, ir))


def test_icl_norm_false_near_the_edge(cuda_device):
    """norm=False: rows of norm up to ~2.6 (e = 2) at tau = 0.4 make the kernels' 1/tau 2.5 * 16 = 40, the limit"""
    B, D = 257, 96
    emb, il, ir = _batch(2 * B + 9, D, B, 13, cuda_device, stress=False)
    g = torch.Generator(device="cuda").manual_seed(14)
    emb = emb / emb.norm(dim=1, keepdim=True) * (1.2 + 1.4 * torch.rand((emb.shape[0], 1), generator=g, device=cuda_device))
    run = _public(0.4, 0.3, il, ir)
    run.norm = False
    _icl_case("norm=False", [emb], il, ir, 0.4, 0.3, [None], run, norm=False)


@pytest.mark.parametrize("inv_tau", [0.25, 2.0, 10.0, 20.0, 40.0, 43.0, 80.0])
def test_icl_anticorrelated_anchor_across_temperatures(cuda_device, inv_tau):
    """Anchor 0 points away from every other row of the batch (its positive included). Beyond the kernels' fixed-maximum
    range every term of its row flushes to zero; such temperatures are refused, and the kernels are shown to fail there."""
    B, D = 200, 64
    emb, il, ir = _batch(2 * B + 9, D, B, 17, cuda_device, anti=True)
    a, b = _operands(emb, il, ir)
    assert float(torch.cat([a[0] @ b.t(), a[0] @ a[1:].t()]).max()) < -0.5
    if inv_tau > sloss.MAX_INV_TAU:
        with pytest.raises(ValueError):
            sloss.icl_loss(tau=1.0 / inv_tau)(emb, torch.stack([il, ir], 1))
        if inv_tau * 1.5 * math.log2(math.e) > 126:        # every s < -0.5: every term of the row flushes to zero
            nll = sloss._IclMany.apply(il, ir, inv_tau, sloss._unsharded(), True, emb)
            assert not bool(torch.isfinite(nll[0, 0, 0])), "the kernels no longer underflow here: revisit MAX_INV_TAU"
        return
    _icl_case(f"anti-correlated 1/tau={inv_tau:g}", [emb], il, ir, 1.0 / inv_tau, 0.5, [None],
              _public(1.0 / inv_tau, 0.5, il, ir))


@pytest.mark.parametrize("B,Ds,Dt,tau,red", [
    (128, 64, 64, 4.0, "mean"), (257, 64, 64, 0.1, "sum"), (300, 300, 1200, 4.0, "sum"), (129, 300, 1200, 0.5, "mean"),
    (1000, 1200, 300, 0.1, "mean"), (256, 1200, 300, 4.0, "sum"), (255, 320, 321, 0.5, "sum"), (2, 320, 321, 0.1, "mean"),
    (3500, 320, 321, 4.0, "mean")])
def test_ial_against_fp64(cuda_device, B, Ds, Dt, tau, red):
    g = torch.Generator(device="cuda").manual_seed(B + Ds + Dt)
    N = 2 * B + 20
    base = torch.randn((N, max(Ds, Dt)), generator=g, device=cuda_device)
    tar = (base[:, :Dt] + 0.3 * torch.randn((N, Dt), generator=g, device=cuda_device)).contiguous()
    src = (base[:, :Ds] + 0.5 * torch.randn((N, Ds), generator=g, device=cuda_device)).contiguous()
    perm = torch.randperm(N, generator=g, device=cuda_device)
    il, ir = perm[:B].contiguous(), perm[B:2 * B].contiguous()
    x = src.clone().requires_grad_(True)
    out = sloss.ial_loss(tau=tau, ab_weight=0.3, zoom=0.1, reduction=red)(x, tar, torch.stack([il, ir], 1))
    out.backward()
    sa, sb = _operands(src, il, ir)
    ta, tb = _operands(tar, il, ir)
    r = ref64.ial_reference(sa, sb, ta, tb, src, il, ir, 1.0 / tau, 0.3, 0.1, red)
    rep = ref64.Report(f"ial {Ds}/{Dt} tau={tau} {red}")
    rep.elementwise("loss", out.detach().reshape(1), torch.tensor([r["loss"]], dtype=torch.float64, device=cuda_device),
                    r["loss_bound"])
    rep.rows("demb", x.grad, r["demb"], r["demb_bound"])
    print(rep)
    rep.check()
