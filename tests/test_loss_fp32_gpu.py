"""GPU: the fp32 route of icl_loss (precision "fp32", snag_b200.loss_fp32) against an fp64 reference whose operands are
the UNROUNDED normalised fp32 rows, anchor by anchor (lse, NLL, loss) and row by row (d emb, d weight_norm), each
against its own bound; plus the kernels of the route on their own and the bf16 route's bitwise invariance.

Error model: that of tests/loss_fp64_reference.py with two terms replaced.
  logits  |ds| <= fp32.tc_margin(Dpad): the tensor cores' measured accumulation error on split operands (per element of
          Dpad, 4x margin), the proven split term 3 * 2^-16 (the dropped m_i m_j and the residuals of the two-term
          splits) and half an fp32 ulp — instead of ops.tc_margin of bf16 operands, whose rounding is part of the operand.
  G       the bf16 route rounds G once (2^-8 |G|). Here G = G_h + G_m + r_G with |r_G| <= 2^-9 |G - G_h| <= 2^-18 |G|,
          and the GEMM against [Y_h ; Y_m ; Y_h] forms G_h Y_h + G_h Y_m + G_m Y_h = (G_h + G_m)(Y_h + Y_m) - G_m Y_m,
          Y_h + Y_m = Y - r_Y, |r_Y| <= 2^-18 |Y|, |G_m Y_m| <= (2^-9 (1 + 2^-8))^2 |G| |Y|: per term
          <= (2^-18 + 2^-18 + 2^-18 (1 + 2^-7)) |G| |Y| < 2^-16 |G| |Y|, i.e. UBF -> 2^-16 in the bound H |Y|.
  The fp32 accumulation of the GEMM keeps its K 2^-23 term (K = 6 Bp adds at most 3x as many terms, all inside |G| |Y|
  with the per-term coefficient above, so the bound's K = 2 Bp term is multiplied by 3).
Every test prints the largest error-to-bound ratio per quantity (run with -s)."""
from __future__ import annotations

import pytest
import torch

from snag_b200 import fp32, loss as sloss, loss_fp32, ops
from tests import loss_fp64_reference as ref64
from tests import test_loss_fp64_gpu as t64

pytestmark = pytest.mark.gpu

SPLIT_G = 2.0 ** -16


def _operands_fp32(emb, il, ir, normalize=True):
    """the unrounded normalised rows the split is made of (fp32.prep's rows: the prologue's arithmetic), in fp64"""
    D = emb.shape[1]
    a = fp32.prep(emb.contiguous(), il, normalize, 0)[0].rows[:, :D].double()
    b = fp32.prep(emb.contiguous(), ir, normalize, 1)[0].rows[:, :D].double()
    return a, b


@pytest.fixture
def fp32_model(monkeypatch):
    """the fp64 reference of tests/loss_fp64_reference.py with the fp32 route's error model and operands, and the
    training switch set to fp32"""
    monkeypatch.setattr(ref64, "eps_logit", lambda d: fp32.tc_margin(ref64.dpad_of(d)))
    monkeypatch.setattr(ref64, "UBF", SPLIT_G)
    monkeypatch.setattr(ref64, "TC_ADD", 3 * 2.0 ** -23)
    monkeypatch.setattr(t64, "_operands", _operands_fp32)
    monkeypatch.setattr(sloss, "TRAIN_PRECISION", "fp32")


ROUTES = [(1, 1, 0.1), (2, 63, 0.1), (127, 64, 0.05), (129, 65, 0.1), (255, 300, 0.1), (257, 321, 0.05),
          (1000, 1200, 0.1), (3500, 1800, 0.1), (3500, 300, 0.05)]


@pytest.mark.parametrize("sym", [True, False])
@pytest.mark.parametrize("B,D,tau", ROUTES)
def test_fp32_route_against_fp64(cuda_device, monkeypatch, fp32_model, B, D, tau, sym):
    """half-Gram forward (sym) or per-side forward, two-kernel split backward; stress rows, weighted table"""
    monkeypatch.setattr(sloss, "SYM_FORWARD", sym)
    emb, il, ir = t64._batch(2 * B + 31, D, B, B * 7 + D, cuda_device)
    g = torch.Generator(device="cuda").manual_seed(B)
    wn = torch.rand((emb.shape[0],), generator=g, device=cuda_device) + 0.5
    t64._icl_case(f"fp32 sym={sym}", [emb], il, ir, tau, 0.3, [wn], t64._public(tau, 0.3, il, ir), saved_e=False)


def test_fp32_forward_many_mixed_widths(cuda_device, fp32_model):
    """18 narrow tables (two 16-table chunks of the prologue and the forward) and two wide ones in one call"""
    B, N = 300, 700
    widths = [64] * 18 + [300, 1200]
    embs, wns = [], []
    _, il, ir = t64._batch(N, 8, B, 11, cuda_device)
    g = torch.Generator(device="cuda").manual_seed(12)
    for p, d in enumerate(widths):
        e = torch.randn((N, d), generator=g, device=cuda_device)
        e[ir] = e[il] + (0.3 + 0.05 * p) * torch.randn((B, d), generator=g, device=cuda_device)
        embs.append(e)
        wns.append(torch.rand((N,), generator=g, device=cuda_device) + 0.5 if p % 3 == 0 else None)
    t64._icl_case("fp32 forward_many", embs, il, ir, 0.1, 0.5, wns, t64._public(0.1, 0.5, il, ir), saved_e=False)


def test_fp32_norm_false(cuda_device, fp32_model):
    """norm=False: rows of norm up to ~2.6 folded into 1/tau by a power of two (exact in fp32)"""
    B, D = 257, 96
    emb, il, ir = t64._batch(2 * B + 9, D, B, 13, cuda_device, stress=False)
    g = torch.Generator(device="cuda").manual_seed(14)
    emb = emb / emb.norm(dim=1, keepdim=True) * (1.2 + 1.4 * torch.rand((emb.shape[0], 1), generator=g, device=cuda_device))
    run = t64._public(0.4, 0.3, il, ir)
    run.norm = False
    t64._icl_case("fp32 norm=False", [emb], il, ir, 0.4, 0.3, [None], run, norm=False, saved_e=False)


@pytest.mark.parametrize("B,D,world,grads", [(1000, 300, 2, "local"), (1000, 300, 2, "gather"), (257, 64, 3, "gather"),
                                             (257, 1200, 3, "local")])
def test_fp32_sharded_against_fp64(cuda_device, fp32_model, B, D, world, grads):
    """anchor-sharded fp32 loss on `world` lock-step ranks (tests/test_loss_fp64_gpu.py's shard)"""
    emb, il, ir = t64._batch(2 * B + 31, D, B, B + D + world, cuda_device)
    g = torch.Generator(device="cuda").manual_seed(world)
    wn = torch.rand((emb.shape[0],), generator=g, device=cuda_device) + 0.5
    t64._icl_case(f"fp32 sharded {grads} w{world}", [emb], il, ir, 0.1, 0.4, [wn],
                  t64._sharded(0.1, 0.4, il, ir, world, grads), saved_e=False)


@pytest.mark.parametrize("B,D", [(1, 1), (129, 63), (300, 300), (257, 1800)])
@pytest.mark.parametrize("normalize", [True, False])
def test_split_prologue_bitwise(cuda_device, B, D, normalize):
    """[m | h | h | m | h] rows of [a ; b ; a]: h bit for bit ops.icl_stack_prep, m bit for bit fp32.prep, zero padding"""
    emb, il, ir = t64._batch(2 * B + 31, D, B, B + D, cuda_device)
    Bp = ops.round_up(B, 256)
    dpad = ops.round_up(D, 64)
    S5 = loss_fp32.icl_stack_prep([emb], il, ir, Bp, normalize)[0]
    S3 = ops.icl_stack_prep([emb], il, ir, Bp, normalize)[0]
    assert tuple(S5.shape) == (3 * Bp, 5 * dpad)
    blk = [S5[:, k * dpad:(k + 1) * dpad] for k in range(5)]
    for k in (1, 2, 4):
        assert torch.equal(blk[k], S3), f"h block {k}"
    assert torch.equal(blk[0], blk[3])
    for part, idx in ((0, il), (1, ir), (2, il)):
        m = fp32.prep(emb, idx, normalize, 0)[0].split[:, :dpad]
        assert torch.equal(blk[0][part * Bp:part * Bp + B], m), f"m of part {part}"
        assert not blk[0][part * Bp + B:(part + 1) * Bp].any()


@pytest.mark.parametrize("B,D,tau", [(300, 300, 0.1), (257, 1200, 0.05)])
def test_split_kernels_against_fp64(cuda_device, B, D, tau):
    """The split half-Gram forward's row sums (lse) and the split dL/dlogits G_h + G_m against fp64 on the fp32 rows"""
    emb, il, ir = t64._batch(2 * B + 31, D, B, 3 * B + D, cuda_device)
    inv_tau = 1.0 / tau
    Bp = ops.round_up(B, 256)
    S5 = loss_fp32.icl_stack_prep([emb], il, ir, Bp)[0]
    a, b = _operands_fp32(emb, il, ir)
    f = ref64.icl_forward(a, b, inv_tau)
    eps_s = fp32.tc_margin(ops.round_up(D, 64))
    eE = (eps_s + 4 * ref64.U32) * inv_tau + ref64.EX2_REL
    stats = loss_fp32.icl_fwd_sym([S5], B, Bp, inv_tau)[0]
    rep = ref64.Report(f"split kernels B={B} D={D}")
    for k, s in ((0, "a"), (2, "b")):
        bound = eE + 2 * B * ref64.U32 + 2 * ref64.U32 * (f[f"lse_{s}"].abs() + inv_tau)
        rep.elementwise("lse", stats[k], f[f"lse_{s}"], bound)
    g = torch.Generator(device="cuda").manual_seed(B)
    ga = (torch.rand((B,), generator=g, device=cuda_device) / B).double()        # dL/dnll of both sides (fp32 values)
    gb = (torch.rand((B,), generator=g, device=cuda_device) / B).double()
    # coefficients from the fp64 lse (rounded to fp32 once), as the backward forms them from the forward's lse
    cra = (ga * torch.exp(inv_tau - f["lse_a"])).float()
    crb = (gb * torch.exp(inv_tau - f["lse_b"])).float()
    dg = (ga + gb).float()
    pad = (lambda t: torch.nn.functional.pad(t, (0, 4 - B % 4)) if B % 4 else t)
    cra, crb, dg = pad(cra).contiguous(), pad(crb).contiguous(), pad(dg).contiguous()
    G3 = loss_fp32.icl_bwd_logits(S5[0:Bp], S5[Bp:3 * Bp], B, Bp, inv_tau, cra, crb, dg)
    assert tuple(G3.shape) == (Bp, 6 * Bp)
    assert torch.equal(G3[:, :2 * Bp], G3[:, 2 * Bp:4 * Bp])
    got = G3[:, :2 * Bp].double() + G3[:, 4 * Bp:].double()
    G, Gabs, dgr = ref64.icl_dlogits(f["Pa"], f["Pb"], ga, gb, inv_tau)
    cols = torch.cat([torch.arange(B, device=cuda_device), Bp + torch.arange(B, device=cuda_device)])
    H = 2.0 ** -17 * G.abs() + (eE + 16 * ref64.U32) * Gabs
    ar = torch.arange(B, device=cuda_device)
    H[ar, ar] += 3 * ref64.U32 * dgr
    rep.elementwise("G_h + G_m", got[:B][:, cols], G, H)
    assert not G3[B:].any() and not got[:B][:, Bp + B:].any() and not got[:B][:, B:Bp].any()
    print(rep)
    rep.check()


def test_fp32_errors_below_bf16(cuda_device, monkeypatch):
    """On the same seeded inputs the fp32 route's largest NLL and d emb errors against the fp64 loss of the unrounded
    rows are below the bf16 route's (printed side by side)"""
    B, D, tau = 3500, 1200, 0.1
    emb, il, ir = t64._batch(2 * B + 31, D, B, 77, cuda_device)
    a, b = _operands_fp32(emb, il, ir)
    r = ref64.icl_reference(a, b, emb, il, ir, 1.0 / tau, 0.5)
    errs = {}
    for prec in ("bf16", "fp32"):
        spy = t64._Spy()
        monkeypatch.setattr(sloss, "_IclMany", spy)
        e = emb.clone().requires_grad_(True)
        out = sloss.icl_loss(tau=tau, ab_weight=0.5).forward_many([e], torch.stack([il, ir], 1), precision=prec)[0]
        out.backward()
        nll = spy.calls[-1][0][0].double()
        e_nll = float(torch.maximum((nll[0] - r["nll_a"]).abs().max(), (nll[1] - r["nll_b"]).abs().max()))
        e_grad = float((e.grad.double() - r["demb"]).norm(dim=1).max() / r["demb"].norm(dim=1).max())
        errs[prec] = (e_nll, e_grad)
    print(f"largest errors against fp64 (NLL abs, d emb rel. to the largest row): bf16 {errs['bf16']}, fp32 {errs['fp32']}, "
          f"ratio {errs['bf16'][0] / errs['fp32'][0]:.1f} / {errs['bf16'][1] / errs['fp32'][1]:.1f}")
    assert errs["fp32"][0] < errs["bf16"][0] and errs["fp32"][1] < errs["bf16"][1]


def _layer_inputs(cuda_device, seed=5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    N, B, dm, M = 900, 300, 64, 4
    mk = lambda w: torch.randn((N, w), generator=g, device=cuda_device).requires_grad_(True)
    streams = [mk(dm) for _ in range(M)] + [None, None]
    hidden = [mk(dm) for _ in range(M)] + [None, None]
    joint, joint_fz = mk(M * dm), mk(M * dm)
    wn = torch.softmax(torch.randn((N, 6), generator=g, device=cuda_device), 1).requires_grad_(True)
    leaves = [t for t in streams + hidden + [joint, joint_fz, wn] if t is not None]
    # every id occurs once in the batch: each gradient row gets one scatter add, so the results are bitwise reproducible
    links = torch.stack([torch.randperm(N // 2, generator=g, device=cuda_device)[:B],
                         N // 2 + torch.randperm(N // 2, generator=g, device=cuda_device)[:B]], 1).to(torch.int32)
    return streams, hidden, joint, joint_fz, wn, leaves, links


def test_fp32_layer_step_graph_capture_bitwise(cuda_device):
    """A SnagLossLayer(precision="fp32") step captured with GraphedStep replays to the eager step's loss and gradients,
    bit for bit"""
    from snag_b200.graphs import GraphedStep
    streams, hidden, joint, joint_fz, wn, leaves, links = _layer_inputs(cuda_device)
    layer = sloss.SnagLossLayer(tau=0.1, ab_weight=0.5, precision="fp32").to(cuda_device)
    fn = lambda: layer(streams, hidden, joint, joint_fz, links, wn)
    step = GraphedStep(fn, leaves + list(layer.parameters()))
    for _ in range(2):
        loss_g = step().clone()
        grads_g = [t.grad.clone() for t in leaves]
        for t in leaves:
            t.grad = None
        loss_e = fn()
        loss_e.backward()
        assert torch.equal(loss_g, loss_e.detach())
        for a_, t in zip(grads_g, leaves):
            assert torch.equal(a_, t.grad)
        for t, a_ in zip(leaves, step.grads):
            t.grad = a_
        links.copy_(links.flip(0).roll(7, 0))


def test_switching_precision_leaves_bf16_bitwise(cuda_device, monkeypatch):
    """bf16 results after an fp32 step (TRAIN_PRECISION switched there and back) equal a fresh bf16 call bit for bit,
    and differ from the fp32 step's"""
    streams, hidden, joint, joint_fz, wn, leaves, links = _layer_inputs(cuda_device, seed=9)

    def step(layer):
        for t in leaves:
            t.grad = None
        out = layer(streams, hidden, joint, joint_fz, links, wn)
        out.backward()
        return out.detach().clone(), [t.grad.clone() for t in leaves]

    fresh = step(sloss.SnagLossLayer(tau=0.1).to(cuda_device))
    layer = sloss.SnagLossLayer(tau=0.1).to(cuda_device)
    monkeypatch.setattr(sloss, "TRAIN_PRECISION", "fp32")
    f32 = step(layer)
    monkeypatch.setattr(sloss, "TRAIN_PRECISION", "bf16")
    again = step(layer)
    assert torch.equal(fresh[0], again[0]) and all(torch.equal(x, y) for x, y in zip(fresh[1], again[1]))
    assert not torch.equal(fresh[0], f32[0])
    assert abs(float(fresh[0]) - float(f32[0])) < 1e-2 * abs(float(f32[0]))
