"""CPU: the fp32 evaluation's host logic. The split bound in fp64; an oracle-built stand-in of snag_b200.fp32 (SplitOperand
tables, exact canonical scores) through the sharded driver (evaluate._align_ranks_steps) under the lockstep simulator and
under gloo, against oracle.align_eval on unrounded fp32 rows; argument checks and refusals; --eval-precision parsing."""
from __future__ import annotations

import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import oracle
from snag_b200 import evaluate, fp32, patch
from snag_b200._lib import SnagError
from tests import oracle_backend as ob


def _split_parts(x):
    h = oracle.bf16_round(x)
    m = oracle.bf16_round((x - h).astype(np.float32))
    return h, m


def _adversarial(n, d, seed):
    rng = np.random.RandomState(seed)
    q = n // 4
    dense = rng.randn(q, d).astype(np.float32) + rng.randn(1, d).astype(np.float32)
    pos = np.abs(rng.randn(q, d)).astype(np.float32)
    wide = (rng.randn(q, d) * np.exp(rng.randn(q, d) * 3)).astype(np.float32)           # wide dynamic range: tiny m
    rest = rng.randn(n - 3 * q, d).astype(np.float32)
    return oracle.normalize_rows(np.concatenate([dense, pos, wide, rest], 0))


@pytest.mark.parametrize("d", [300, 1200])
def test_split_bound(d):
    """|x - h - m| <= 2^-16 |x| per element and |x.y - (m_x h_y + h_x m_y + h_x h_y)| <= 3 * 2^-16 * sum |x_k y_k| per
    pair (fp64 throughout): the split term of fp32.tc_margin."""
    x = _adversarial(512, d, 1)
    h, m = _split_parts(x)
    xd, hd, md = x.astype(np.float64), h.astype(np.float64), m.astype(np.float64)
    assert (np.abs(xd - hd - md) <= 2.0 ** -16 * np.abs(xd)).all()
    exact = xd @ xd.T
    split = md @ hd.T + hd @ md.T + hd @ hd.T
    absum = np.abs(xd) @ np.abs(xd).T
    ratio = np.abs(exact - split) / np.maximum(absum, 1e-300)
    assert ratio.max() <= fp32.SPLIT_REL_ERR, ratio.max()
    assert fp32.tc_margin(1216) > fp32.SPLIT_REL_ERR + 4 * fp32.FP32_TC_DOT_ERR_PER_K * 1216


def _operand(x, side):
    """A host SplitOperand of unrounded rows x (the layout snag_prep_split writes) and ||row||^2 as oracle.norm2."""
    n, d = x.shape
    dpad = evaluate.round_up(d, 64)
    rows = np.zeros((n, dpad), np.float32)
    rows[:, :d] = x
    h, m = _split_parts(rows)
    parts = [h, m, h] if side else [m, h, h]
    split = torch.from_numpy(np.concatenate(parts, 1)).to(torch.bfloat16)
    return fp32.SplitOperand(split, torch.from_numpy(rows)), torch.from_numpy(oracle.norm2(x))


def _rows(t):
    return t.rows if isinstance(t, fp32.SplitOperand) else t


def _wrap(f):
    return lambda *a, **kw: f(*[_rows(v) for v in a], **{k: _rows(v) for k, v in kw.items()})


# the stand-in of snag_b200.fp32: the oracle backend's exact scores on the fp32 rows the SplitOperands carry
backend = types.SimpleNamespace(
    eval_rowtopk=_wrap(ob.eval_rowtopk), topk_merge_mean=ob.topk_merge_mean, topk_rescore=_wrap(ob.topk_rescore),
    pair_score=_wrap(ob.pair_score), eval_rank=_wrap(ob.eval_rank), top4_merge=ob.top4_merge,
    top3_rescore=_wrap(ob.top3_rescore), num_sms=lambda: 148, LAST_TOPK_INFO={}, LAST_RANK_INFO={})


def _problem(n, d, seed):
    rng = np.random.RandomState(seed)
    x = oracle.normalize_rows(rng.randn(n, d).astype(np.float32))
    y = oracle.normalize_rows((x + 0.7 * rng.randn(n, d)).astype(np.float32))
    assert not np.array_equal(oracle.bf16_round(x), x)                  # genuinely fp32 rows
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
    x, y = _problem(300, 48, 31 + world)              # 300 targets over 8 ranks: ranks 2..7 own nothing
    (X, xn), (Y, yn) = _operand(x, 0), _operand(y, 1)
    res = evaluate.simulate_sharded(
        lambda r: evaluate._align_ranks_steps(backend, X, Y, xn, yn, 300, k, csls, True, world, r), world)
    ref = oracle.align_eval(x, y, csls, k)
    for r in res:
        _check(r, ref, csls)


def test_split_operand_plumbing():
    x, _ = _problem(40, 70, 2)
    X, _ = _operand(x, 0)
    assert X.shape == (40, 128) and X.split.shape == (40, 384)
    sub = X[5:9]
    assert torch.equal(sub.rows, X.rows[5:9]) and torch.equal(sub.split, X.split[5:9])
    ids = torch.tensor([3, 0, 39])
    g = X.index_select(0, ids)
    assert torch.equal(g.rows, X.rows[ids]) and torch.equal(g.split, X.split[ids])
    with pytest.raises(ValueError):
        fp32.SplitOperand(X.split[:, :128], X.rows)


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
    x, y = _problem(300, 48, 6)
    (X, xn), (Y, yn) = _operand(x, 0), _operand(y, 1)
    gen = evaluate._align_ranks_steps(backend, X, Y, xn, yn, 300, 10, True, True, world, rank)
    res = evaluate._drive_with_torch_distributed(gen, dist.group.WORLD)
    try:
        _check(res, oracle.align_eval(x, y, True, 10), True)
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


def test_argument_checks_and_refusals():
    emb = torch.zeros((40, 8))
    left, right = torch.arange(0, 20), torch.arange(20, 40)
    with pytest.raises(ValueError, match="precision"):
        evaluate.evaluate_alignment(emb, left, right, precision="fp16")
    with pytest.raises(SnagError, match="csls_k=17"):
        evaluate.evaluate_alignment(emb, left, right, csls=True, csls_k=17, precision="fp32")
    with pytest.raises(SnagError, match="GPU"):
        evaluate.evaluate_alignment(emb, left, right, csls=True, csls_k=10, precision="fp32")
    with pytest.raises(SnagError, match="bf16 operands only"):
        evaluate.evaluate_alignment_host(emb[:20], emb[20:], 20, precision="fp32")
    with pytest.raises(ValueError, match="precision"):
        evaluate.evaluate_alignment_host(emb[:20], emb[20:], 20, precision="tf32")
    with pytest.raises(SnagError):                                  # host tensors never reach a kernel
        fp32.prep(emb, None, True, 0)
    assert evaluate.EVAL_PRECISION == "bf16"                        # the trainer's default


def test_eval_precision_flag_parsing():
    assert patch.parse_args(["/ref", "--csls", "--csls_k", "3"]) == (None, "/ref", ["--csls", "--csls_k", "3"])
    assert patch.parse_args(["--eval-precision", "fp32", "/ref", "--epochs", "2"]) == ("fp32", "/ref", ["--epochs", "2"])
    assert patch.parse_args(["--eval-precision=bf16", "/ref"]) == ("bf16", "/ref", [])
    # main.py's own arguments are left alone, whatever they are called
    assert patch.parse_args(["/ref", "--eval-precision", "fp32"]) == (None, "/ref", ["--eval-precision", "fp32"])
    for bad in (["--eval-precision", "fp64", "/ref"], ["--eval-precision"], ["--eval-precision", "fp32"]):
        with pytest.raises(SystemExit):
            patch.parse_args(bad)


def test_patch_sets_the_trainer_precision(monkeypatch):
    monkeypatch.setattr(evaluate, "EVAL_PRECISION", "bf16")
    patch.patch(eval_precision="fp32")
    assert evaluate.EVAL_PRECISION == "fp32"
    patch.patch()                                                   # None leaves it as it is
    assert evaluate.EVAL_PRECISION == "fp32"
    with pytest.raises(ValueError):
        patch.patch(eval_precision="half")
    patch.unpatch()


def test_runner_passes_the_precision(monkeypatch):
    from snag_b200 import runner
    seen = {}

    def fake(final_emb, test_left, test_right, **kw):
        seen.update(kw)
        raise StopIteration                                         # the metrics tail is not under test here

    monkeypatch.setattr(evaluate, "evaluate_alignment", fake)
    monkeypatch.setattr(evaluate, "EVAL_PRECISION", "fp32")
    model = types.SimpleNamespace(joint_emb_generat=lambda: (torch.zeros((4, 8)), None))
    args = types.SimpleNamespace(model_name="SNAG", distance=2, csls=True, csls_k=3)
    with pytest.raises(StopIteration):
        runner._test(types.SimpleNamespace(model=model, args=args), torch.arange(2), torch.arange(2, 4))
    assert seen["precision"] == "fp32"
