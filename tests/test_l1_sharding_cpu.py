"""CPU: the fused --distance 1 evaluation's host logic. An oracle-built stand-in of snag_b200.l1 runs the sharded driver
(evaluate._align_ranks_steps, three-sweep path) under the lockstep simulator and under gloo; the streaming and audit
references of tests/l1_reference.py against oracle.align_eval_l1; argument checks of evaluate_alignment_l1."""
from __future__ import annotations

import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import oracle
from snag_b200 import evaluate
from snag_b200._lib import SnagError
from tests import l1_reference
from tests.conftest import golden_names, load_golden

KT = 16


def _np(t):
    return t.detach().cpu().float().numpy()


def _dist(X, Y, nv1, nv2, n1, n2, use_csls):
    d = oracle.l1_distance(_np(X[:n1]), _np(Y[:n2]))
    if not use_csls:
        return d
    return l1_reference._chain(d, _np(nv1)[:n1, None], _np(nv2)[None, :n2])


def _eval_rowtopk(X, Y, xn, yn, n1, n2, want_idx=False):
    c = (np.float32(1.0) - oracle.l1_distance(_np(X[:n1]), _np(Y[:n2]))).astype(np.float32)
    part = np.full((1, n1, KT), -np.inf, np.float32)
    pidx = np.full((1, n1, KT), -1, np.int32)
    kk = min(KT, n2)
    order = np.lexsort((-np.broadcast_to(np.arange(n2), c.shape), c), axis=1)[:, -kk:]
    part[0, :, KT - kk:] = np.take_along_axis(c, order, 1)
    pidx[0, :, KT - kk:] = order
    return (torch.from_numpy(part), torch.from_numpy(pidx)) if want_idx else torch.from_numpy(part)


def _topk_merge_mean(part, k, want_nv=True, want_cand=False, part_idx=None):
    allv = np.concatenate(list(part.numpy()), axis=1)
    alli = np.concatenate(list(part_idx.numpy()), axis=1)
    order = np.lexsort((-alli, allv), axis=1)[:, -KT:]
    return None, torch.from_numpy(np.take_along_axis(allv, order, 1).copy()), torch.from_numpy(
        np.take_along_axis(alli, order, 1).astype(np.int32))


def _topk_rescore(A, B, an, bn, cand_idx, cand_val, k, n_b, tag="rows", outsider_bound=None):
    v = np.sort(cand_val.numpy(), axis=1)[:, ::-1]
    return torch.from_numpy(l1_reference._mean_desc(v[:, :k], k))


def _pair_score(X, Y, n, xn, yn, nv1, nv2, use_csls):
    d = np.diag(oracle.l1_distance(_np(X[:n]), _np(Y[:n]))).astype(np.float32)
    return torch.from_numpy(l1_reference._chain(d, _np(nv1)[:n], _np(nv2)[:n]) if use_csls else d)


def _eval_rank(X, Y, xn, yn, nv1, nv2, g_row, g_col, row_gid0, col_gid0, n1, n2, use_csls, cnt_row, cnt_col, want_top3=False):
    dist = _dist(X, Y, nv1, nv2, n1, n2, use_csls)
    gr, gc = _np(g_row)[:n1], _np(g_col)[:n2]
    ri = row_gid0 + np.arange(n1)[:, None]
    cj = col_gid0 + np.arange(n2)[None, :]
    same = ri == cj
    prow = ((dist < gr[:, None]) | ((dist == gr[:, None]) & (cj < ri))) & ~same
    pcol = ((dist < gc[None, :]) | ((dist == gc[None, :]) & (ri < cj))) & ~same
    cnt_row[:n1] += torch.from_numpy(prow.sum(1).astype(np.int32))
    cnt_col[:n2] += torch.from_numpy(pcol.sum(0).astype(np.int32))
    if not want_top3:
        return None, None
    order = np.lexsort((np.broadcast_to(cj, dist.shape), dist), axis=1)[:, :4]
    v = np.full((1, n1, 4), -np.inf, np.float32)
    i = np.full((1, n1, 4), 0x7FFFFFFF, np.int32)
    v[0, :, :order.shape[1]] = -np.take_along_axis(dist, order, 1)
    i[0, :, :order.shape[1]] = order + col_gid0
    return torch.from_numpy(v), torch.from_numpy(i)


def _top4_merge(val, idx):
    v = np.concatenate(list(val.numpy()), axis=1)
    i = np.concatenate(list(idx.numpy()), axis=1)
    order = np.lexsort((i, -v), axis=1)[:, :4]
    return torch.from_numpy(np.take_along_axis(v, order, 1)), torch.from_numpy(np.take_along_axis(i, order, 1))


def _top3_rescore(X, Y, xn, yn, nv1, nv2, use_csls, cand):
    dist = _dist(X, Y, nv1, nv2, cand.shape[0], Y.shape[0], use_csls)
    ci = cand.numpy().astype(np.int64)
    ok = ci != 0x7FFFFFFF
    v = np.where(ok, np.take_along_axis(dist, np.where(ok, ci, 0), 1), np.inf).astype(np.float32)
    order = np.lexsort((ci, v), axis=1)
    return torch.from_numpy(np.take_along_axis(v, order, 1)), torch.from_numpy(np.take_along_axis(ci, order, 1).astype(np.int32))


# the stand-in of snag_b200.l1: exact (oracle) scores, the same entry points and list layouts
backend = types.SimpleNamespace(
    eval_rowtopk=_eval_rowtopk, topk_merge_mean=_topk_merge_mean, topk_rescore=_topk_rescore, pair_score=_pair_score,
    eval_rank=_eval_rank, top4_merge=_top4_merge, top3_rescore=_top3_rescore, num_sms=lambda: 148,
    LAST_TOPK_INFO={}, LAST_RANK_INFO={})


def _operands(x, y):
    X = torch.from_numpy(np.ascontiguousarray(x, np.float32))
    Y = torch.from_numpy(np.ascontiguousarray(y, np.float32))
    return X, Y, X.abs().sum(1), Y.abs().sum(1), x.shape[0]


def _problem(n, d, seed):
    rng = np.random.RandomState(seed)
    x = oracle.normalize_rows(rng.randn(n, d).astype(np.float32))
    y = oracle.normalize_rows((x + 0.7 * rng.randn(n, d)).astype(np.float32))
    return x, y


def _check(res, ref, csls):
    np.testing.assert_array_equal(res.rank_l2r.numpy(), ref["rank_l2r"])
    np.testing.assert_array_equal(res.rank_r2l.numpy(), ref["rank_r2l"])
    np.testing.assert_array_equal(res.g.numpy(), ref["g"])
    np.testing.assert_array_equal(res.top3_idx.numpy(), ref["top3"])
    if csls:
        np.testing.assert_array_equal(res.nv1.numpy(), ref["nv1"])
        np.testing.assert_array_equal(res.nv2.numpy(), ref["nv2"])


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("csls,k", [(True, 10), (True, 3), (False, 1)])
def test_simulated_shards_match_the_oracle(world, csls, k):
    x, y = _problem(300, 48, 17 + world)               # 300 targets over 8 ranks: ranks 2..7 own nothing
    X, Y, xn, yn, n = _operands(x, y)
    res = evaluate.simulate_sharded(
        lambda r: evaluate._align_ranks_steps(backend, X, Y, xn, yn, n, k, csls, True, world, r, two_sweep=False), world)
    ref = oracle.align_eval_l1(x, y, csls, k)
    for r in res:
        _check(r, ref, csls)


@pytest.mark.parametrize("name", golden_names("l1_"))
def test_goldens_through_the_driver(name):
    fx = load_golden(name)
    X, Y, xn, yn, n = _operands(fx["x"], fx["y"])
    res = evaluate.simulate_sharded(
        lambda r: evaluate._align_ranks_steps(backend, X, Y, xn, yn, n, int(fx["k"]), bool(fx["csls"]), True, 2, r,
                                              two_sweep=False), 2)
    np.testing.assert_array_equal(res[1].rank_l2r.numpy(), fx["rank_l2r"])
    np.testing.assert_array_equal(res[0].rank_r2l.numpy(), fx["rank_r2l"])
    np.testing.assert_array_equal(res[0].top3_idx.numpy(), fx["top3"])


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    x, y = _problem(300, 48, 5)
    X, Y, xn, yn, n = _operands(x, y)
    gen = evaluate._align_ranks_steps(backend, X, Y, xn, yn, n, 10, True, True, world, rank, two_sweep=False)
    res = evaluate._drive_with_torch_distributed(gen, dist.group.WORLD)
    ref = oracle.align_eval_l1(x, y, True, 10)
    try:
        _check(res, ref, True)
        out[rank] = True
    except AssertionError:
        out[rank] = False
    dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_gloo_world2_matches_the_oracle():
    last = None
    for _attempt in range(2):          # the rendezvous port is picked optimistically; retry once if it was taken meanwhile
        try:
            with mp.Manager() as mgr:
                out = mgr.dict()
                mp.spawn(_gloo_worker, args=(2, _free_port(), out), nprocs=2, join=True)
                assert dict(out) == {0: True, 1: True}
                return
        except AssertionError:
            raise
        except Exception as e:         # rendezvous / socket errors
            last = e
    raise last


@pytest.mark.parametrize("csls,k,block", [(True, 10, 64), (True, 16, 1000), (False, 1, 37)])
def test_streaming_reference_matches_align_eval_l1(csls, k, block):
    x, y = _problem(257, 33, 3)
    ref = oracle.align_eval_l1(x, y, csls, k)
    got = l1_reference.align_eval_l1_stream(x, y, csls, k, block_rows=block)
    for f in ("rank_l2r", "rank_r2l", "g") + (("nv1", "nv2") if csls else ()):
        np.testing.assert_array_equal(got[f], ref[f], err_msg=f)


@pytest.mark.parametrize("csls", [True, False])
def test_audit_reference_matches_align_eval_l1(csls):
    x, y = _problem(220, 40, 9)
    ref = oracle.align_eval_l1(x, y, csls, 7)
    sel = np.array([0, 5, 99, 219])
    a = l1_reference.audit_l1(x[sel], y, sel, csls, 7, ref.get("nv2"), False)
    np.testing.assert_array_equal(a["rank"], ref["rank_l2r"][sel])
    np.testing.assert_array_equal(a["g"], ref["g"][sel])
    b = l1_reference.audit_l1(y[sel], x, sel, csls, 7, ref.get("nv1"), True)
    np.testing.assert_array_equal(b["rank"], ref["rank_r2l"][sel])
    if csls:
        np.testing.assert_array_equal(a["nv"], ref["nv1"][sel])
        np.testing.assert_array_equal(b["nv"], ref["nv2"][sel])


def test_argument_checks():
    emb = torch.zeros((8, 4))
    left, right = torch.arange(0, 4), torch.arange(4, 8)
    with pytest.raises(ValueError, match="pair up"):
        evaluate.evaluate_alignment_l1(emb, left, torch.arange(4, 7))
    with pytest.raises(ValueError, match="exceeds"):
        evaluate.evaluate_alignment_l1(emb, left, right, csls=True, csls_k=5)
    with pytest.raises(SnagError, match="GPU"):
        evaluate.evaluate_alignment_l1(emb, left, right, csls=True, csls_k=2)


def test_large_k_with_a_group_is_refused():
    emb = torch.zeros((40, 4))
    with pytest.raises(SnagError, match="not sharded"):
        evaluate.evaluate_alignment_l1(emb, torch.arange(0, 20), torch.arange(20, 40), csls=True, csls_k=17, group=object())
