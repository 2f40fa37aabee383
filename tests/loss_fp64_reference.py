"""fp64 reference of the contrastive losses (model/SNAG_loss.py:58-128 and 148-202) on the bf16 operands the kernels
consume, with a per-element error bound derived from the kernels' arithmetic, and a comparator that checks every
anchor's lse / NLL and every embedding-gradient row against its own bound.

Operands. `a`, `b` are the rows the tensor cores see (bf16 values held in fp64): for icl_loss the normalised rows
emb[idx_l], emb[idx_r] rounded once to bf16 (the output of the prologue kernel). Gradients reach `emb` through the
backward of F.normalize of the fp32 rows (a straight-through estimator: value = the rounded rows), as in the reference.

Error model (u32 = 2^-24, ubf = 2^-8 the unit roundoff of bf16, K = 2 Bp the contraction length of the gradient GEMM):
  logits      |ds| <= eps_s = ops.tc_margin(Dpad)          (the measured tensor-core dot error, 4x margin, of unit rows)
  E = ex2((s - 1) log2e / tau): relative  eps_E = (eps_s + 4 u32) / tau + EX2_REL
  row sum     n - 1 <= 2B fp32 additions of positive terms: relative 2B u32
  lse         eps_lse = eps_E + 2B u32 + 2 u32 (|lse| + 1/tau)
  NLL         eps_nll = eps_lse + eps_s / tau + u32 (|nll| + |lse|)
  G = dL/dlogits, rounded once to bf16 (the recomputing backward) or E and then G (the saved-E backward):
              |dG_ij| <= ubf |G_ij| (+ ubf Gabs_ij with saved E) + (eps_E + eps_nll + 8 u32) Gabs_ij
                         + 3 u32 (Gabs_ij + [cross diagonal] dg_i / tau)
              with Gabs_ij = (c_i P_ij + c'_j P'_ji) / tau the softmax parts of G without the -1 of the positives
  dz = G . Y  |ddz_ik| <= sum_j |dG_ij| |Y_jk| + K 2^-23 sum_j |G_ij| |Y_jk|   (fp32 accumulation, one unit per add)
  d emb       ||d demb_e|| <= sum over occurrences of (||ddz_i||_2 + (D + 4) u32 ||dz_i||_2) / ||emb_e||
                              + (m_e - 1) u32 sum_i ||dz_i||_2 / ||emb_e||   (m_e occurrences scattered with atomics)
ial_loss: the kernel rounds the ebar-centred matrices Gs, Gt and their difference to bf16 (loss.py:559-576), so |G| is
taken on those values, and the coefficient errors act on |E - ebar| + ebar (both the centred part and the part added
back in fp32)."""
from __future__ import annotations

import math

import torch

from snag_b200 import ops

U32 = 2.0 ** -24
UBF = 2.0 ** -8
EX2_REL = 2.0 ** -22           # PTX ISA: ex2.approx.f32, maximum relative error 2^-22 over the full range
TC_ADD = 2.0 ** -23            # one unit of fp32 rounding per tensor-core accumulation step
MASK = float("-inf")


def round_bf16(t: torch.Tensor) -> torch.Tensor:
    """fp64 -> nearest bf16 value (via fp32, as the kernels round fp32 values), back in fp64"""
    return t.float().to(torch.bfloat16).double()


def dpad_of(d: int) -> int:
    return ops.round_up(d, 64)


def eps_logit(d: int) -> float:
    return ops.tc_margin(dpad_of(d))


def eps_e(d: int, inv_tau: float) -> float:
    return (eps_logit(d) + 4 * U32) * inv_tau + EX2_REL


def _sides(a: torch.Tensor, b: torch.Tensor, inv_tau: float):
    """fp64 logits of both sides, [cross | self] with the self diagonal masked: La = [a b^T | a a^T], Lb = [b a^T | b b^T]"""
    n = a.shape[0]
    eye = torch.eye(n, dtype=torch.bool, device=a.device)
    sab = a @ b.t()
    La = torch.cat([sab, (a @ a.t()).masked_fill(eye, MASK)], 1) * inv_tau
    Lb = torch.cat([sab.t(), (b @ b.t()).masked_fill(eye, MASK)], 1) * inv_tau
    return La, Lb


def icl_forward(a: torch.Tensor, b: torch.Tensor, inv_tau: float) -> dict:
    """Per-anchor lse and NLL of both sides (fp64) and the row softmaxes."""
    La, Lb = _sides(a, b, inv_tau)
    lse_a, lse_b = torch.logsumexp(La, 1), torch.logsumexp(Lb, 1)
    pos = (a * b).sum(1) * inv_tau
    return dict(lse_a=lse_a, lse_b=lse_b, nll_a=lse_a - pos, nll_b=lse_b - pos,
                Pa=torch.exp(La - lse_a[:, None]), Pb=torch.exp(Lb - lse_b[:, None]))


def icl_dlogits(Pa, Pb, c_row, c_col, inv_tau, fault=None):
    """dL/dlogits of one side as the kernels lay it out: row i carries every term of dL/d(anchor i).
    Pa: this side's softmax [B, 2B], Pb: the other side's; c_row / c_col: dL/dnll of this / the other side, [B].
      cross: G_ij = (c_i Pa_ij + c'_j Pb_ji) / tau - [i == j] (c_i + c'_i) / tau
      self : G_ij = (c_i Pa_ij + c_j Pa_ji) / tau
    Returns (G, Gabs, dg) with Gabs the same without the positives' -1 and dg = (c_i + c'_i) / tau.
    fault (planted faults for the comparator's own tests): {"drop_diag": i} leaves out anchor i's cross-diagonal entry,
    {"drop_col": j} leaves anchor j out of the column (transposed-role) terms."""
    n = c_row.numel()
    fault = fault or {}
    c_self_col = c_row
    if "drop_col" in fault:
        c_col, c_self_col = c_col.clone(), c_row.clone()
        c_col[fault["drop_col"]] = 0.0
        c_self_col[fault["drop_col"]] = 0.0
    cross = c_row[:, None] * Pa[:, :n] + (c_col[:, None] * Pb[:, :n]).t()
    self_ = c_row[:, None] * Pa[:, n:] + (c_self_col[:, None] * Pa[:, n:]).t()
    Gabs = torch.cat([cross, self_], 1) * inv_tau
    dg = (c_row + c_col) * inv_tau
    G = Gabs.clone()
    ar = torch.arange(n, device=G.device)
    G[ar, ar] -= dg
    if "drop_diag" in fault:
        G[fault["drop_diag"], fault["drop_diag"]] = 0.0
    return G, Gabs, dg


def normalize_bwd(emb: torch.Tensor, idx: torch.Tensor, dz: torch.Tensor, norm: bool = True, scale: float = 1.0):
    """Rows of d emb contributed by dz through gather + F.normalize (fp64), [B, D]; norm=False: the power-of-two scale"""
    if not norm:
        return dz * scale
    e = emb.double()[idx]
    r = e.norm(dim=1, keepdim=True).clamp_min(1e-12)
    z = e / r
    return (dz - z * (z * dz).sum(1, keepdim=True)) / r


def icl_reference(a, b, emb, idx_l, idx_r, inv_tau, ab_weight, w=None, norm=True, scale=1.0, saved_e=False,
                  fault=None) -> dict:
    """The reference op sequence of icl_loss on the operands a, b ([B, D] bf16 values), its gradients and their bounds.
    w: the per-pair weights min(w[l], w[r]) ([B], or None); the loss is sum_i w_i (alpha nll_a + (1 - alpha) nll_b) / B.
    emb: the fp32 table the rows came from (for the normalise backward); scale: 2^-e of norm=False.
    saved_e: bound of the backward that forms G from the forward's bf16 E.
    fault: planted faults for the comparator's own tests ({"drop_diag": i} or {"drop_col": j}).
    Returns fp64 tensors: lse/nll of both sides with their bounds, loss, dz_a/dz_b [B, D] with elementwise bounds,
    demb [N, D] with a row bound [N], and the per-pair d loss / d w [B] with its bound."""
    a, b = a.double(), b.double()
    n, d = a.shape
    fault = fault or {}
    w = torch.ones(n, dtype=torch.float64, device=a.device) if w is None else w.double()
    f = icl_forward(a, b, inv_tau)
    ca, cb = ab_weight * w / n, (1 - ab_weight) * w / n
    out = dict(f)
    eE = eps_e(d, inv_tau)
    out["lse_bound_a"] = eE + 2 * n * U32 + 2 * U32 * (f["lse_a"].abs() + inv_tau)
    out["lse_bound_b"] = eE + 2 * n * U32 + 2 * U32 * (f["lse_b"].abs() + inv_tau)
    for s in "ab":
        out[f"nll_bound_{s}"] = out[f"lse_bound_{s}"] + eps_logit(d) * inv_tau + U32 * (f[f"nll_{s}"].abs() + f[f"lse_{s}"].abs())
    eps_nll = float(torch.maximum(out["nll_bound_a"].max(), out["nll_bound_b"].max()))
    terms = w * (ab_weight * f["nll_a"] + (1 - ab_weight) * f["nll_b"]) / n
    out["loss"] = terms.sum()
    out["loss_bound"] = float((w * (ab_weight * out["nll_bound_a"] + (1 - ab_weight) * out["nll_bound_b"])).sum() / n) \
        + 2 * n * U32 * float(terms.abs().sum())
    out["dw"] = (ab_weight * f["nll_a"] + (1 - ab_weight) * f["nll_b"]) / n
    out["dw_bound"] = (ab_weight * out["nll_bound_a"] + (1 - ab_weight) * out["nll_bound_b"]) / n + 4 * U32 * out["dw"].abs()
    K = 2 * ops.round_up(n, 256)
    for side, (P_this, P_other, c_this, c_other, Y) in (("a", (f["Pa"], f["Pb"], ca, cb, torch.cat([b, a], 0))),
                                                          ("b", (f["Pb"], f["Pa"], cb, ca, torch.cat([a, b], 0)))):
        side_fault = {k: v for k, v in fault.items() if k == "drop_col" or side == "a"}
        G, Gabs, dg = icl_dlogits(P_this, P_other, c_this, c_other, inv_tau, side_fault)
        H = UBF * G.abs() + ((UBF if saved_e else 0.0) + eE + eps_nll + 11 * U32) * Gabs
        ar = torch.arange(n, device=G.device)
        H[ar, ar] += 3 * U32 * dg
        Ya = Y.abs()
        out[f"dz_{side}"] = G @ Y
        out[f"dz_bound_{side}"] = H @ Ya + K * TC_ADD * (G.abs() @ Ya)
    _emb_rows(out, emb, idx_l, idx_r, norm, scale, d)
    return out


def _emb_rows(out, emb, idx_l, idx_r, norm, scale, d):
    """d emb and its per-row bound from dz_a / dz_b and their elementwise bounds"""
    N = emb.shape[0]
    dev = out["dz_a"].device
    demb = torch.zeros((N, d), dtype=torch.float64, device=dev)
    bound = torch.zeros((N,), dtype=torch.float64, device=dev)
    mass = torch.zeros((N,), dtype=torch.float64, device=dev)
    count = torch.zeros((N,), dtype=torch.float64, device=dev)
    inv_r = (1.0 / emb.double().norm(dim=1).clamp_min(1e-12)) if norm else torch.full((N,), scale, dtype=torch.float64,
                                                                                       device=dev)
    for idx, s in ((idx_l, "a"), (idx_r, "b")):
        dz, dzb = out[f"dz_{s}"], out[f"dz_bound_{s}"]
        demb.index_add_(0, idx, normalize_bwd(emb, idx, dz, norm, scale))
        dzn = dz.norm(dim=1)
        bound.index_add_(0, idx, (dzb.norm(dim=1) + ((d + 4) * U32 if norm else 0.0) * dzn) * inv_r[idx])
        mass.index_add_(0, idx, dzn * inv_r[idx])
        count.index_add_(0, idx, torch.ones_like(dzn))
    out["demb"] = demb
    out["demb_bound"] = bound + (count - 1).clamp_min(0) * U32 * mass


def dw_table(ref: dict, wl: torch.Tensor, wr: torch.Tensor, idx_l: torch.Tensor, idx_r: torch.Tensor, N: int):
    """d loss / d weight_norm through min(w[l], w[r]) (the first minimum on ties, as torch.min), and its bound"""
    to_l = wl <= wr
    tgt = torch.where(to_l, idx_l, idx_r)
    dev = ref["dw"].device
    g = torch.zeros((N,), dtype=torch.float64, device=dev).index_add_(0, tgt, ref["dw"])
    gb = torch.zeros((N,), dtype=torch.float64, device=dev).index_add_(0, tgt, ref["dw_bound"])
    cnt = torch.zeros((N,), dtype=torch.float64, device=dev).index_add_(0, tgt, torch.ones_like(ref["dw"]))
    return g, gb + cnt * U32 * g.abs()


# ------------------------------------------------------------------------------------------------ IAL
def ial_reference(src_a, src_b, tar_a, tar_b, emb, idx_l, idx_r, inv_tau, ab_weight, zoom, reduction) -> dict:
    """ial_loss (model/SNAG_loss.py:148-202): zoom (alpha KL(Q_a || P_a) + (1 - alpha) KL(Q_b || P_b)) reduced by `mean`
    over the [B, 2B] matrix or by `sum`, with P from the source rows, Q from the (detached) target rows. Returns the
    loss with its bound and d emb (the source table) with a row bound."""
    sa, sb, ta, tb = (t.double() for t in (src_a, src_b, tar_a, tar_b))
    n, ds = sa.shape
    dt = ta.shape[1]
    fs, ft = icl_forward(sa, sb, inv_tau), icl_forward(ta, tb, inv_tau)
    denom = 2.0 * n * n if reduction == "mean" else 1.0
    g_a, g_b = zoom * ab_weight / denom, zoom * (1 - ab_weight) / denom
    out = {}
    eEs, eEt = eps_e(ds, inv_tau), eps_e(dt, inv_tau)
    e_lse = max(eEs, eEt) + 2 * n * U32
    La_s, Lb_s = _sides(sa, sb, inv_tau)
    La_t, Lb_t = _sides(ta, tb, inv_tau)
    K = 2 * ops.round_up(n, 256)
    loss, loss_bound = 0.0, 0.0
    for g, s, Ls, Lt in ((g_a, "a", La_s, La_t), (g_b, "b", Lb_s, Lb_t)):
        Q = ft[f"P{s}"]
        fin = torch.isfinite(Ls)
        ls, lt = Ls.masked_fill(~fin, 0.0), Lt.masked_fill(~fin, 0.0)
        kl = (Q * (lt - ls)).sum(1) - ft[f"lse_{s}"] + fs[f"lse_{s}"]
        loss = loss + g * float(kl.sum())
        # Q rounded to bf16 once (plus its own logit / lse errors), contracted with both tables, 1/tau-scaled dots
        lse_terms = 2 * (e_lse + 2 * U32 * (float(fs[f"lse_{s}"].abs().max()) + inv_tau))
        row = ((UBF + eEt + e_lse + 8 * U32) * (Q * (lt - ls).abs()).sum(1) + lse_terms
               + (K * TC_ADD + max(ds, dt) * U32) * inv_tau * 2 * (1 + 2 ** -7)
               + 4 * U32 * (kl.abs() + fs[f"lse_{s}"].abs() + ft[f"lse_{s}"].abs()))
        loss_bound += g * float(row.sum())
    out["loss"] = loss
    out["loss_bound"] = loss_bound + 2 * n * U32 * abs(loss)
    ebar = math.exp(-inv_tau)
    eps_c = max(eEs, eEt) + e_lse + 8 * U32
    ar = torch.arange(n, device=sa.device)
    for side, (Ps, Po_s, Pt, Po_t, c_row, c_col, Y) in (
            ("a", (fs["Pa"], fs["Pb"], ft["Pa"], ft["Pb"], g_a, g_b, torch.cat([sb, sa], 0))),
            ("b", (fs["Pb"], fs["Pa"], ft["Pb"], ft["Pa"], g_b, g_a, torch.cat([sa, sb], 0)))):
        cr = torch.full((n,), c_row, dtype=torch.float64, device=sa.device)
        cc = torch.full((n,), c_col, dtype=torch.float64, device=sa.device)
        _, Ms, _ = icl_dlogits(Ps, Po_s, cr, cc, inv_tau)
        _, Mt, _ = icl_dlogits(Pt, Po_t, cr, cc, inv_tau)
        G = Ms - Mt                                       # no positives' -1 in a KL: the diagonal terms cancel
        # the kernel's values: coefficient (cr_i + cc_j) / tau times (E_ij - ebar), E = P exp(lse - 1/tau)
        coef_s, coef_t = _coef(cr, cc, fs, side, inv_tau), _coef(cr, cc, ft, side, inv_tau)
        Es, Et = _e_matrix(sa, sb, side, inv_tau), _e_matrix(ta, tb, side, inv_tau)
        Gs_c, Gt_c = coef_s * (Es - ebar), coef_t * (Et - ebar)
        Mag = coef_s * ((Es - ebar).abs() + ebar) + coef_t * ((Et - ebar).abs() + ebar)
        for t in (Gs_c, Gt_c, Mag):                       # the masked self diagonal is written as 0
            t[:, n:][ar, ar] = 0.0
        H = UBF * (Gs_c.abs() + Gt_c.abs() + (Gs_c - Gt_c).abs()) + eps_c * Mag
        Ya = Y.abs()
        out[f"dz_{side}"] = G @ Y
        out[f"dz_bound_{side}"] = H @ Ya + K * TC_ADD * (Mag @ Ya)
    _emb_rows(out, emb, idx_l, idx_r, True, 1.0, ds)
    return out


def _e_matrix(a, b, side, inv_tau):
    """E = exp((s - 1) / tau) over [cross | self] of one side, 0 on the masked diagonal"""
    x, y = (a, b) if side == "a" else (b, a)
    n = x.shape[0]
    E = torch.exp((torch.cat([x @ y.t(), x @ x.t()], 1) - 1.0) * inv_tau)
    E[:, n:][torch.arange(n), torch.arange(n)] = 0.0
    return E


def _coef(cr_g, cc_g, f, side, inv_tau):
    """(cr_i + cc_j) / tau of EpiIclBwd with cr_i = g exp(1/tau - lse_i) of this side, cc_j of the other side (cross)
    or this side (self)"""
    other = "b" if side == "a" else "a"
    cr = cr_g * torch.exp(inv_tau - f[f"lse_{side}"])
    cc = cc_g * torch.exp(inv_tau - f[f"lse_{other}"])
    return torch.cat([cr[:, None] + cc[None, :], cr[:, None] + cr[None, :]], 1) * inv_tau


# ------------------------------------------------------------------------------------------------ comparator
class Report:
    """Largest |got - ref| / bound per quantity; `check` raises when any ratio exceeds 1."""

    def __init__(self, route: str):
        self.route, self.ratios, self.where = route, {}, {}

    def elementwise(self, name, got, ref, bound):
        got, ref = got.double().to(ref.device), ref.double()
        bound = torch.as_tensor(bound, dtype=torch.float64, device=ref.device).expand_as(ref)
        err = (got - ref).abs()
        err = torch.where(torch.isfinite(got), err, torch.full_like(err, float("inf")))
        ratio = err / bound
        ratio = torch.where((err == 0) & (bound == 0), torch.zeros_like(ratio), ratio)
        self._note(name, ratio)

    def rows(self, name, got, ref, bound):
        """row-wise 2-norm of the error against a bound per row"""
        got, ref = got.double().to(ref.device), ref.double()
        err = (got - ref).norm(dim=-1)
        err = torch.where(torch.isfinite(got).all(-1), err, torch.full_like(err, float("inf")))
        ratio = torch.where((err == 0) & (bound == 0), torch.zeros_like(err), err / bound)
        self._note(name, ratio)

    def _note(self, name, ratio):
        ratio = ratio.reshape(-1)
        k = int(torch.argmax(torch.nan_to_num(ratio, nan=float("inf"))))
        r = float(ratio[k]) if not math.isnan(float(ratio[k])) else float("inf")
        if r >= self.ratios.get(name, -1.0):
            self.ratios[name], self.where[name] = r, k

    def worst(self) -> float:
        return max(self.ratios.values()) if self.ratios else 0.0

    def __str__(self):
        return f"{self.route}: " + ", ".join(f"{k} {v:.3g} (at {self.where[k]})" for k, v in sorted(self.ratios.items()))

    def check(self):
        assert self.worst() <= 1.0, f"error exceeds the bound: {self}"
        return self
