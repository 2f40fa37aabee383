"""The link-precision switch without a GPU: `python -m snag_b200.patch --link-precision`, patch(link_precision=), the
drop-ins reading mining.LINK_PRECISION, and the refusals of mining / seeds, which come before anything reaches a device."""
from __future__ import annotations

import types

import pytest
import torch

from snag_b200 import SnagError, evaluate, fp32, mining, ops, patch, seeds


def test_link_precision_flag_parsing():
    assert patch.parse_args(["--link-precision", "fp32", "/ref", "--epochs", "2"]) == (None, "/ref", ["--epochs", "2"])
    assert patch.parse_args(["--link-precision", "fp32", "/ref"]).link_precision == "fp32"
    assert patch.parse_args(["--link-precision=bf16", "/ref"]).link_precision == "bf16"
    assert patch.parse_args(["/ref", "--csls"]).link_precision is None
    for argv in (["--eval-precision", "fp32", "--link-precision", "bf16", "/ref", "--il"],
                 ["--link-precision", "bf16", "--eval-precision=fp32", "/ref", "--il"]):
        opts = patch.parse_args(argv)
        assert opts == ("fp32", "/ref", ["--il"])
        assert opts.link_precision == "bf16"
    # after the reference directory everything is main.py's
    opts = patch.parse_args(["/ref", "--link-precision", "fp32"])
    assert opts == (None, "/ref", ["--link-precision", "fp32"]) and opts.link_precision is None
    for bad in (["--link-precision", "fp16", "/ref"], ["--link-precision"], ["--link-precision", "fp32"],
                ["--link-precision=", "/ref"], ["--eval-precision", "fp32", "--link-precision"],
                ["--link-precision", "fp32", "--eval-precision", "tf32", "/ref"]):
        with pytest.raises(SystemExit):
            patch.parse_args(bad)


def test_patch_sets_the_link_precision(monkeypatch):
    monkeypatch.setattr(mining, "LINK_PRECISION", "bf16")
    monkeypatch.setattr(evaluate, "EVAL_PRECISION", "bf16")
    patch.patch(eval_precision="fp32")                              # the evaluation's switch leaves the links alone
    assert mining.LINK_PRECISION == "bf16" and evaluate.EVAL_PRECISION == "fp32"
    patch.patch(link_precision="fp32")
    assert mining.LINK_PRECISION == "fp32" and evaluate.EVAL_PRECISION == "fp32"
    patch.patch()                                                   # None leaves both as they are
    assert mining.LINK_PRECISION == "fp32"
    with pytest.raises(ValueError):
        patch.patch(link_precision="fp16")
    with pytest.raises(ValueError):                                 # nothing is set when one value is refused
        patch.patch(eval_precision="bf16", link_precision="half")
    assert evaluate.EVAL_PRECISION == "fp32"
    patch.unpatch()


def test_trainer_default_is_bf16():
    assert mining.LINK_PRECISION == "bf16"


def test_iter_new_links_drop_in_reads_the_switch(monkeypatch):
    seen = []
    monkeypatch.setattr(mining, "iter_new_links", lambda *a, **kw: seen.append(kw["precision"]) or [])
    fake = types.SimpleNamespace(args=types.SimpleNamespace(semi_learn_step=5))
    for p in ("fp32", "bf16"):
        monkeypatch.setattr(mining, "LINK_PRECISION", p)
        mining.Iter_new_links(fake, 4, [0], torch.zeros((2, 8)), [1])
    assert seen == ["fp32", "bf16"]


def test_refusals_come_before_the_device():
    x, y = torch.randn((6, 8)), torch.randn((5, 8))                 # host tensors: a kernel call would raise SnagError
    for bad in ("fp16", "tf32", "FP32"):
        with pytest.raises(ValueError, match="precision"):
            mining.mutual_nearest(x, y, precision=bad)
        with pytest.raises(ValueError, match="precision"):
            mining.iter_new_links([0], [1], x, [], True, precision=bad)
        with pytest.raises(ValueError, match="precision"):
            seeds.topk_similarity_entries(x, y, 3, precision=bad)
    with pytest.raises(ValueError, match="canonical=False"):
        mining.mutual_nearest(x, y, canonical=False, precision="fp32")
    for p in ("bf16", "fp32"):                                      # valid arguments reach the C ABI and fail there
        with pytest.raises(SnagError):
            mining.mutual_nearest(x, y, precision=p)
        with pytest.raises(SnagError):
            seeds.topk_similarity_entries(x, y, 3, precision=p)


def test_admission_margin_comes_from_the_error_model():
    pool_kth = torch.tensor(0.8)
    # bf16 at the image widths: at or below the fixed 4e-6 the sweep used before, so it admits a superset
    for dpad in (2048, 4096):
        eps = ops.tc_margin(dpad, 1.0)
        assert eps >= 7.4e-5
        assert float(seeds._admission_threshold(pool_kth, eps)) <= 0.8 - 4e-6
        # fp32 adds the split term: a wider margin than bf16 at the same width
        assert fp32.tc_margin(dpad, 1.0) > eps
    assert float(seeds._admission_threshold(pool_kth, 1e-4)) == pytest.approx(0.8 - 4e-4)
