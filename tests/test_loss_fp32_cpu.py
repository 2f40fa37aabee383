"""CPU: the training-precision switch of icl_loss (loss.TRAIN_PRECISION, forward_many(precision=),
SnagLossLayer(precision=), patch(train_precision=), --train-precision), its refusals, and the host algebra of the fp32
route — split stacks, windows, the [G_h | G_h | G_m] backward — with a torch-CPU stand-in for the loss_fp32 entry points,
unsharded against the reference's golden loss and under real torch.distributed (gloo) at worlds 2 and 3."""
from __future__ import annotations

import os

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from snag_b200 import loss as sloss
from snag_b200 import patch as sp
from tests import oracle_backend as ob
from tests.conftest import load_golden
from tests.test_loss_sharding_cpu import _free_port, _problem, _run


# ------------------------------------------------------------------------------------------------ CPU stand-in
class SplitStandIn:
    """torch-CPU stand-in for snag_b200.loss_fp32 on the same split-stack layout ([3 Bp, 5 Dpad] bf16 rows
    [m | h | h | m | h]); the contractions are taken on h + m in fp32 (the kernels' m_i h_j + h_i m_j + h_i h_j differs
    by m_i m_j <= 2^-16, far below what these tests compare)."""

    @staticmethod
    def icl_stack_prep(embs, idx_l, idx_r, Bp, normalize=True):
        out = []
        for e in embs:
            n, d = idx_l.numel(), e.shape[1]
            dpad = ob.round_up(d, 64)
            S = torch.zeros((3 * Bp, 5 * dpad), dtype=torch.bfloat16)
            for part, idx in ((0, idx_l), (1, idx_r), (2, idx_l)):
                z = e.index_select(0, idx)
                z = torch.nn.functional.normalize(z, dim=1) if normalize else z
                h = z.to(torch.bfloat16)
                m = (z - h.float()).to(torch.bfloat16)
                rows = slice(part * Bp, part * Bp + n)
                for k, t in enumerate((m, h, h, m, h)):
                    S[rows, k * dpad:k * dpad + d] = t
            out.append(S)
        return out

    @staticmethod
    def rows(S):
        """h + m of the rows (fp32), from the side-0 window"""
        dpad = S.shape[1] // 5
        return S[:, dpad:2 * dpad].float() + S[:, :dpad].float()

    @classmethod
    def icl_fwd_sym(cls, S5s, B, Bp, inv_tau, rank=0, world=1, all_reduce=None):
        return ob.icl_fwd_sym([cls.rows(S) for S in S5s], B, Bp, inv_tau, rank, world, all_reduce)

    @classmethod
    def icl_side(cls, X, Y, B, Bp, inv_tau, row0=0, nx=None):
        return ob.icl_side(cls.rows(X), cls.rows(Y), B, Bp, inv_tau, row0, nx)

    @classmethod
    def icl_bwd_logits(cls, X, Y, B, Bp, inv_tau, cr, cc, dg, row0=0, nx=None):
        """G in fp32 as oracle_backend.icl_bwd_logits forms it, stored as [G_h | G_h | G_m]"""
        nx = Bp if nx is None else nx
        s, dead, gr = ob._icl_logits(cls.rows(X), cls.rows(Y), B, Bp, inv_tau, row0, nx)
        E = torch.exp(s * inv_tau - inv_tau)
        ok = gr < B
        pad = lambda t: torch.cat([t[:B], torch.zeros(Bp - B)])
        crp, ccp, dgp = pad(cr), pad(cc), pad(dg)
        cr_i = torch.where(ok, crp[gr.clamp(max=Bp - 1)], torch.zeros(()))
        G = (cr_i[:, None] + torch.cat([ccp, crp])[None, :]) * E * inv_tau
        i = torch.arange(nx)[ok]
        G[i, gr[ok]] -= dgp[gr[ok]] * inv_tau
        G = G.masked_fill(dead, 0.0)
        G[~ok] = 0.0
        Gh = G.to(torch.bfloat16)
        return torch.cat([Gh, Gh, (G - Gh.float()).to(torch.bfloat16)], 1)

    @staticmethod
    def grad_contract_rows(G3, Yrows, n_rows, d, keep_parts=False):
        dpad = Yrows.shape[1] // 5
        Y3 = torch.cat([Yrows[:, 2 * dpad:3 * dpad], Yrows[:, 3 * dpad:4 * dpad], Yrows[:, 4 * dpad:]], 0)   # [Y_h ; Y_m ; Y_h]
        return G3[:n_rows].float() @ Y3[:, :d].float()

    normalize_bwd_scatter = staticmethod(ob.normalize_bwd_scatter)


def _crit(tau=0.1, group=None, grads="gather"):
    crit = sloss.icl_loss(tau=tau, ab_weight=0.4, n_view=2)
    if group is None:
        crit.shard = sloss.AnchorShard(be=ob)
    else:
        crit.distribute(group, grads=grads, be=ob)
    crit.fp32_be = SplitStandIn
    return crit


# ------------------------------------------------------------------------------------------------ switch and options
def test_options_parse_train_precision_in_any_order():
    o = sp.parse_args(["--train-precision", "fp32", "--eval-precision=fp32", "/ref", "--data", "x"])
    assert tuple(o) == ("fp32", "/ref", ["--data", "x"]) and o.train_precision == "fp32" and o.link_precision is None
    o = sp.parse_args(["--link-precision=fp32", "--train-precision=bf16", "/ref"])
    assert tuple(o) == (None, "/ref", []) and o.train_precision == "bf16" and o.link_precision == "fp32"
    o = sp.parse_args(["/ref", "--train-precision", "fp32"])         # after the directory: main.py's argument
    assert o.train_precision is None and o[2] == ["--train-precision", "fp32"]
    assert len(o) == 3
    for bad in (["--train-precision", "fp16", "/ref"], ["--train-precision"], ["--train-precision=tf32", "/ref"]):
        with pytest.raises(SystemExit):
            sp.parse_args(bad)


def test_patch_sets_and_refuses_train_precision(monkeypatch):
    monkeypatch.setattr(sloss, "TRAIN_PRECISION", "bf16")
    with pytest.raises(ValueError):
        sp.patch(train_precision="fp16")
    assert sloss.TRAIN_PRECISION == "bf16"
    try:
        sp.patch(train_precision="fp32")
        assert sloss.TRAIN_PRECISION == "fp32"
    finally:
        sp.unpatch()


def test_unknown_precisions_are_refused_before_any_device_call(monkeypatch):
    emb, links, wn = _problem(40, 16, 100, 3)          # CPU tensors: any kernel call would raise SnagError instead
    crit = sloss.icl_loss(tau=0.1)
    with pytest.raises(ValueError, match="precision"):
        crit.forward_many([emb], links, precision="fp16")
    with pytest.raises(ValueError, match="precision"):
        sloss.SnagLossLayer(precision="tf32")
    monkeypatch.setattr(sloss, "TRAIN_PRECISION", "fp64")
    with pytest.raises(ValueError, match="precision"):
        crit(emb, links)


def test_default_is_bf16_and_read_at_call_time(monkeypatch):
    assert sloss.TRAIN_PRECISION == "bf16" and sloss.SnagLossLayer().precision is None
    emb, links, wn = _problem(64, 24, 200, 4)
    crit = _crit()
    l_bf16 = _run(crit, emb, links, wn)[0]
    monkeypatch.setattr(sloss, "TRAIN_PRECISION", "fp32")
    l_fp32 = _run(crit, emb, links, wn)[0]
    monkeypatch.setattr(sloss, "TRAIN_PRECISION", "bf16")
    assert torch.equal(_run(crit, emb, links, wn)[0], l_bf16) and not torch.equal(l_fp32, l_bf16)


# ------------------------------------------------------------------------------------------------ host algebra
def test_stand_in_fp32_route_matches_reference_golden(monkeypatch):
    """the fp32 host algebra (windows, G3, K-stacked rows) reproduces the reference's fp32 loss and gradients far more
    closely than the bf16 route's 5e-3 / 2e-2"""
    fx = load_golden("icl_tau0.1_w")
    crit = sloss.icl_loss(tau=float(fx["tau"]), ab_weight=float(fx["ab_weight"]), n_view=2)
    crit.shard = sloss.AnchorShard(be=ob)
    crit.fp32_be = SplitStandIn
    monkeypatch.setattr(sloss, "TRAIN_PRECISION", "fp32")
    for sym in (True, False):
        monkeypatch.setattr(sloss, "SYM_FORWARD", sym)
        out, g, gw = _run(crit, torch.from_numpy(fx["emb"]), fx["links"], torch.from_numpy(fx["weight_norm"]))
        np.testing.assert_allclose(out.item(), float(fx["loss"]), rtol=1e-4)
        gref = torch.from_numpy(fx["grad_emb"])
        assert float((g - gref).norm() / gref.norm()) < 1e-3


def _worker(rank, world, port, B, D, grads, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    sloss.TRAIN_PRECISION = "fp32"
    emb, links, wn = _problem(B, D, 2 * B + 50, 7)
    ref = _run(_crit(), emb, links, wn)
    loss, g, gw = _run(_crit(group=dist.group.WORLD, grads=grads), emb, links, wn)
    if grads == "local":
        dist.all_reduce(g)
    ok = (abs(loss.item() - ref[0].item()) < 1e-5 and float((g - ref[1]).abs().max()) < 1e-5 * float(ref[1].abs().max() + 1)
          and float((gw - ref[2]).abs().max()) < 1e-5)
    out[rank] = bool(ok)
    dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world,B,D,grads", [(2, 300, 48, "gather"), (2, 130, 32, "local"), (3, 200, 40, "gather"),
                                             (3, 257, 40, "local")])
def test_gloo_sharded_fp32_equals_unsharded(world, B, D, grads):
    last = None
    for _attempt in range(2):
        try:
            with mp.Manager() as mgr:
                out = mgr.dict()
                mp.spawn(_worker, args=(world, _free_port(), B, D, grads, out), nprocs=world, join=True)
                assert dict(out) == {r: True for r in range(world)}
                return
        except AssertionError:
            raise
        except Exception as e:
            last = e
    raise last
