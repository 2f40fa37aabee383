"""The drop-in boundary: signatures of the mirrors equal the reference's (checked against the unmodified reference tree:
baseline/_ref on the GPU box, /root/reference in the build container), patch() rebinds every name main.py / model/SNAG.py use, and Runner._test
reproduces the reference's log lines, CSV and side effects (GPU)."""
from __future__ import annotations

import inspect
import logging
import math
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import oracle

from baseline import harness, install_ref

REF = harness.ref_root()
needs_ref = pytest.mark.skipif(REF is None, reason="no reference checkout on this machine (baseline/install_ref.py)")


def test_installed_reference_is_unmodified():
    """baseline/_ref (what the GPU box and bench.py import) holds exactly the reference's files: the manifest written
    at install time still matches, and — where /root/reference is present — so does the original."""
    if not os.path.isdir(install_ref.DST):
        pytest.skip("baseline/_ref not installed")
    assert install_ref.verify()
    if os.path.isdir(install_ref.SRC):
        assert install_ref._digests(install_ref.SRC) == install_ref._digests(install_ref.DST)


def _sig(f):
    """Parameter names, kinds and defaults (annotations do not matter to a caller)."""
    return [(p.name, p.kind, p.default) for p in inspect.signature(f).parameters.values()]


@needs_ref
def test_loss_weighting_layers_equal_the_reference_classes():
    """CustomMultiLossLayer (evaluated on stacked tensors here) and AutomaticWeightedLoss against the reference's own
    classes on CPU: value and gradients, with the int 0 an absent modality contributes (model/SNAG.py:147-160), with a
    short list, and the state-dict keys the optimiser groups by (src/utils.py:46-54)."""
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    from refshim import load_reference
    ref = load_reference()
    import importlib
    from snag_b200 import loss
    torch.manual_seed(0)
    for entries in ([0.7, 1.3, 0, 0.2], [2.0, 0, 0, 0, 0.5, 1.0], [0.4], [0, 0]):
        mine, theirs = loss.CustomMultiLossLayer(loss_num=6), ref.loss.CustomMultiLossLayer(loss_num=6)
        assert list(mine.state_dict().keys()) == list(theirs.state_dict().keys()) == ["log_vars"]
        lv = torch.randn(6)
        with torch.no_grad():
            mine.log_vars.copy_(lv)
            theirs.log_vars.copy_(lv)
        outs = []
        for layer in (mine, theirs):
            ls = [torch.tensor(float(v), requires_grad=True) if v != 0 else 0 for v in entries]
            out = layer(ls)
            out.backward()
            outs.append((out.item(), layer.log_vars.grad.clone(), [l.grad.item() for l in ls if isinstance(l, torch.Tensor)]))
        np.testing.assert_allclose(outs[0][0], outs[1][0], rtol=1e-6)
        np.testing.assert_allclose(outs[0][1].numpy(), outs[1][1].numpy(), rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(outs[0][2], outs[1][2], rtol=1e-6)
    awl_ref = importlib.import_module("model.Tool_model").AutomaticWeightedLoss(7)
    awl = loss.AutomaticWeightedLoss(7)
    assert list(awl.state_dict().keys()) == list(awl_ref.state_dict().keys())
    xs = [torch.tensor(v) for v in (0.3, 1.1, 2.0)]
    np.testing.assert_allclose(awl(*xs).item(), awl_ref(*xs).item(), rtol=1e-6)


@needs_ref
def test_signatures_match_reference():
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    from refshim import load_reference
    ref = load_reference()
    import importlib
    from snag_b200 import evaluate, loss, mining, noise
    for name in ("icl_loss", "ial_loss", "CustomMultiLossLayer"):
        r, m = getattr(ref.loss, name), getattr(loss, name)
        assert _sig(r.__init__) == _sig(m.__init__), name
        assert _sig(r.forward) == _sig(m.forward), name
    assert _sig(ref.utils.pairwise_distances) == _sig(evaluate.pairwise_distances)
    assert _sig(ref.utils.csls_sim) == _sig(evaluate.csls_sim)
    ref_snag = importlib.import_module("model.SNAG").SNAG
    for name in ("add_noise_to_embeddings", "get_mean_std", "update_noise"):
        assert _sig(getattr(ref_snag, name)) == _sig(getattr(noise, name)), name
    assert _sig(ref_snag.Iter_new_links) == _sig(mining.Iter_new_links)
    enc = importlib.import_module("model.SNAG_tools").MultiModalEncoder
    assert _sig(enc.forward) == _sig(noise.encoder_forward)
    from snag_b200 import fusion
    assert _sig(importlib.import_module("model.SNAG_tools").MformerFusion.forward) == _sig(fusion.MformerFusion_forward)
    from snag_b200 import seeds
    assert _sig(importlib.import_module("src.data").visual_pivot_induction) == _sig(seeds.visual_pivot_induction)


def test_signatures_match_the_recorded_reference_signatures():
    """Without a reference checkout: the call signatures SURVEY.md §(a) recorded from the reference (model/SNAG_loss.py,
    src/utils.py:202,417, main.py:359) — parameter names, order and defaults — against the mirrors."""
    from snag_b200 import evaluate, loss, runner
    P = inspect.Parameter.POSITIONAL_OR_KEYWORD
    E = inspect.Parameter.empty
    recorded = {
        loss.icl_loss.forward: [("self", E), ("emb", E), ("train_links", E), ("neg_l", None), ("neg_r", None),
                                ("weight_norm", None), ("norm", True)],
        loss.ial_loss.forward: [("self", E), ("src_emb", E), ("tar_emb", E), ("train_links", E), ("norm", True)],
        evaluate.pairwise_distances: [("x", E), ("y", None)],
        evaluate.csls_sim: [("sim_mat", E), ("k", E)],
        runner._test: [("self", E), ("test_left", E), ("test_right", E), ("last_epoch", False), ("save_name", ""),
                       ("loss", None)],
    }
    for f, want in recorded.items():
        assert _sig(f) == [(n, P, d) for n, d in want], f.__qualname__


@needs_ref
def test_patch_rebinds_reference_names(monkeypatch):
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    from refshim import load_reference
    load_reference()
    import importlib
    from snag_b200 import evaluate, loss, noise, patch, runner
    mods = {n: importlib.import_module(n) for n in ("model.SNAG_loss", "model.SNAG", "model.SNAG_tools", "src.utils", "src.data")}
    saved = {(n, k): v for n, m in mods.items() for k, v in vars(m).items()}
    snag_cls, enc_cls = mods["model.SNAG"].SNAG, mods["model.SNAG_tools"].MultiModalEncoder
    fus_cls = mods["model.SNAG_tools"].MformerFusion
    saved_cls = {(c, k): c.__dict__[k] for c in (snag_cls, enc_cls, fus_cls) for k in
                 ("add_noise_to_embeddings", "get_mean_std", "update_noise", "Iter_new_links", "forward") if k in c.__dict__}
    fake_main = types.ModuleType("main")
    fake_main.Runner = type("Runner", (), {"_test": lambda self: None})
    try:
        done = patch.patch(fake_main)
        assert mods["model.SNAG"].icl_loss is loss.icl_loss and mods["model.SNAG_loss"].ial_loss is loss.ial_loss
        assert mods["src.utils"].pairwise_distances is evaluate.pairwise_distances
        assert mods["model.SNAG"].pairwise_distances is evaluate.pairwise_distances
        assert snag_cls.update_noise is noise.update_noise and enc_cls.forward is noise.encoder_forward
        from snag_b200 import mining
        assert snag_cls.Iter_new_links is mining.Iter_new_links
        assert fake_main.Runner._test is runner._test and fake_main.csls_sim is evaluate.csls_sim
        from snag_b200 import fusion
        assert fus_cls.forward is fusion.MformerFusion_forward
        from snag_b200 import seeds
        assert mods["src.data"].visual_pivot_induction is seeds.visual_pivot_induction
        assert len(done) >= 14
    finally:
        assert patch.unpatch() == len(done)
    # unpatch() put every original back
    for (n, k), v in saved.items():
        assert getattr(mods[n], k) is v, (n, k)
    for (c, k), v in saved_cls.items():
        assert c.__dict__[k] is v, (c, k)
    assert not hasattr(fake_main, "csls_sim")


class _Capture(logging.Handler):
    def __init__(self):
        super().__init__()
        self.lines = []

    def emit(self, record):
        self.lines.append(record.getMessage())


@pytest.mark.gpu
def test_runner_test_mirror(cuda_device, tmp_path):
    from snag_b200 import runner
    rng = np.random.RandomState(3)
    N, n, d = 900, 400, 128
    emb = rng.randn(N, d).astype(np.float32)
    left = rng.permutation(N // 2)[:n]
    right = N // 2 + rng.permutation(N // 2)[:n]
    emb[right] = emb[left] + 0.9 * rng.randn(n, d).astype(np.float32)
    emb_t = torch.from_numpy(emb).to(cuda_device)

    class FakeModel(torch.nn.Module):
        def joint_emb_generat(self):
            return emb_t, None

    logger = logging.getLogger("snag_test_runner")
    logger.setLevel(logging.INFO)
    cap = _Capture()
    logger.addHandler(cap)
    acc_hist = [0.0]
    me = types.SimpleNamespace(
        args=types.SimpleNamespace(model_name="SNAG", distance=2, csls=True, csls_k=3, data_path=str(tmp_path),
                                   data_choice="DBP15K", w_name=False, w_char=False),
        model=FakeModel(), logger=logger, loss_item=0.1234, epoch=7, early_stop_count=5, early_stop_init=50,
        loss_log=types.SimpleNamespace(acc=acc_hist, update_acc=lambda v: acc_hist.append(v)), best_model_wts=None)
    tl, tr = torch.from_numpy(left).to(cuda_device), torch.from_numpy(right).to(cuda_device)
    runner._test(me, tl, tr, last_epoch=False)
    x = oracle.bf16_round(oracle.normalize_rows(emb[left]))
    y = oracle.bf16_round(oracle.normalize_rows(emb[right]))
    ref = oracle.align_eval(x, y, True, 3)
    m = oracle.metrics(ref["rank_l2r"])
    mr = oracle.metrics(ref["rank_r2l"])
    # the device normalisation may round a handful of elements differently from numpy: compare the formatted lines
    want_l2r = f"Ep 7 | l2r: acc of top [1, 10, 50] = {m['acc']}, mr = {m['mr']:.3f}, mrr = {m['mrr']:.3f}, Loss = 0.1234"
    want_r2l = f"Ep 7 | r2l: acc of top [1, 10, 50] = {mr['acc']}, mr = {mr['mr']:.3f}, mrr = {mr['mrr']:.3f}, Loss = 0.1234"
    assert cap.lines[0] == want_l2r and cap.lines[1] == want_r2l
    assert cap.lines[2].startswith("Best model update in Ep 7: MRR from [0.0] --> [")
    assert me.early_stop_count == 50 and len(acc_hist) == 2 and me.best_model_wts is not None
    # last epoch: Res line + prediction CSV, no best-model update
    cap.lines.clear()
    runner._test(me, tl, tr, last_epoch=True, save_name="unit")
    assert cap.lines[2] == f"Res:[{m['acc'][0]}\t{m['acc'][1]}\t{m['mrr']:.3f}]"
    assert me.early_stop_count == 49
    rows = open(os.path.join(str(tmp_path), "SNAG", "unit_pred", "DBP15K_pred.txt")).read().strip().splitlines()
    assert rows[0] == "idx,rank,query_id,gt_id,ret1,ret2,ret3" and len(rows) == n + 1
    got = np.array([[int(v) for v in r.split(",")] for r in rows[1:]])
    assert (got[:, 1] == ref["rank_l2r"]).mean() > 0.99
    assert (got[:, 2] == left).all() and (got[:, 3] == right).all()
    assert (got[:, 4:7] == right[ref["top3"]]).mean() > 0.99


@needs_ref
@pytest.mark.parametrize("name", ["fusion_m4_d64", "fusion_m6_d96"])
def test_mformer_fusion_mirror_on_cpu(monkeypatch, name):
    """The drop-in MformerFusion.forward (snag_b200.fusion) run on the reference's own module instance (weights restored
    from the golden file) reproduces what the reference's forward returned — with the CUDA tail replaced by the oracle's
    restatement, so that the mirrored control flow around the reference's transformer layers is checked on the CPU."""
    import io
    import types as _types
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    from refshim import load_reference
    load_reference()
    import importlib
    from snag_b200 import fusion
    from tests.conftest import load_golden
    fx = load_golden(name)
    M, D, heads = int(fx["M"]), int(fx["D"]), int(fx["heads"])
    tools = importlib.import_module("model.SNAG_tools")
    args = _types.SimpleNamespace(num_hidden_layers=1, num_attention_heads=heads, hidden_size=D, intermediate_size=2 * D,
                                  use_intermediate=1)
    mod = tools.MformerFusion(args, modal_num=M, with_weight=1)
    mod.load_state_dict(torch.load(io.BytesIO(fx["state"].tobytes())))
    mod.eval()

    def cpu_tail(embs, weight_norm, weight_norm_fz):
        j, jf = oracle.joint_fuse([e.detach().numpy() for e in embs], weight_norm.detach().numpy(),
                                  weight_norm_fz.detach().numpy())
        return torch.from_numpy(j), torch.from_numpy(jf)
    monkeypatch.setattr(fusion, "joint_embeddings", cpu_tail)
    embs = [torch.from_numpy(fx[f"emb{m}"]) for m in range(M)] + [None] * (6 - M)
    with torch.no_grad():
        joint, joint_fz, hidden, weight_norm = fusion.MformerFusion_forward(mod, embs)
    np.testing.assert_allclose(weight_norm.numpy(), fx["weight_norm"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(hidden.numpy(), fx["hidden"], rtol=0, atol=1e-5)
    np.testing.assert_allclose(joint.numpy(), fx["joint"], rtol=0, atol=2e-6)
    np.testing.assert_allclose(joint_fz.numpy(), fx["joint_fz"], rtol=0, atol=2e-6)


class _BertSelfAttention(torch.nn.Module):
    def __init__(self, D):
        super().__init__()
        self.query, self.key, self.value = torch.nn.Linear(D, D), torch.nn.Linear(D, D), torch.nn.Linear(D, D)


class _DenseNorm(torch.nn.Module):
    def __init__(self, d_in, D):
        super().__init__()
        self.dense, self.LayerNorm = torch.nn.Linear(d_in, D), torch.nn.LayerNorm(D, eps=1e-12)


class _BertLayer(torch.nn.Module):
    """A BERT encoder layer (post-LayerNorm, eps 1e-12, erf GELU) under the parameter names of the reference's
    fusion_layer. With the weights stored in the fusion golden files it reproduces the hidden states the reference
    recorded there exactly, so it can stand in for the reference's layer where no reference checkout exists."""

    def __init__(self, D, heads):
        super().__init__()
        self.heads = heads
        self.attention = torch.nn.Module()
        self.attention.self, self.attention.output = _BertSelfAttention(D), _DenseNorm(D, D)
        self.intermediate = torch.nn.Module()
        self.intermediate.dense = torch.nn.Linear(D, 2 * D)
        self.output = _DenseNorm(2 * D, D)

    def forward(self, x, output_attentions=False):
        N, M, D = x.shape
        sa, hd = self.attention.self, D // self.heads
        split = lambda t: t.view(N, M, self.heads, hd).permute(0, 2, 1, 3)
        q, k, v = split(sa.query(x)), split(sa.key(x)), split(sa.value(x))
        probs = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(hd), dim=-1)
        ctx = (probs @ v).permute(0, 2, 1, 3).reshape(N, M, D)
        a = self.attention.output.LayerNorm(self.attention.output.dense(ctx) + x)
        y = self.output.LayerNorm(self.output.dense(torch.nn.functional.gelu(self.intermediate.dense(a))) + a)
        return (y, probs) if output_attentions else (y,)


@pytest.mark.parametrize("name", ["fusion_m4_d64", "fusion_m6_d96"])
def test_mformer_fusion_mirror_on_recorded_reference_outputs(monkeypatch, name):
    """Without a reference checkout: the drop-in MformerFusion.forward, run on a module that carries the reference
    module's stored weights (fusion_layer through _BertLayer, weight_raw), reproduces the outputs the reference's forward
    recorded in the golden file, with the CUDA tail replaced by the oracle's restatement as in the test above."""
    import io
    from snag_b200 import fusion
    from tests.conftest import load_golden
    fx = load_golden(name)
    M, D, heads = int(fx["M"]), int(fx["D"]), int(fx["heads"])
    mod = torch.nn.Module()
    mod.args = types.SimpleNamespace(num_attention_heads=heads)
    mod.fusion_layer = torch.nn.ModuleList([_BertLayer(D, heads)])
    mod.weight_raw = torch.nn.Parameter(torch.zeros(6))
    mod.load_state_dict(torch.load(io.BytesIO(fx["state"].tobytes())), strict=True)
    mod.eval()

    def cpu_tail(embs, weight_norm, weight_norm_fz):
        j, jf = oracle.joint_fuse([e.detach().numpy() for e in embs], weight_norm.detach().numpy(),
                                  weight_norm_fz.detach().numpy())
        return torch.from_numpy(j), torch.from_numpy(jf)
    monkeypatch.setattr(fusion, "joint_embeddings", cpu_tail)
    embs = [torch.from_numpy(fx[f"emb{m}"]) for m in range(M)] + [None] * (6 - M)
    with torch.no_grad():
        joint, joint_fz, hidden, weight_norm = fusion.MformerFusion_forward(mod, embs)
    np.testing.assert_allclose(weight_norm.numpy(), fx["weight_norm"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(hidden.numpy(), fx["hidden"], rtol=0, atol=1e-5)
    np.testing.assert_allclose(joint.numpy(), fx["joint"], rtol=0, atol=2e-6)
    np.testing.assert_allclose(joint_fz.numpy(), fx["joint_fz"], rtol=0, atol=2e-6)
