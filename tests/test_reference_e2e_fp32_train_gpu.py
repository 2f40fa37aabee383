"""GPU integration of the fp32 training route with the UNMODIFIED reference (baseline/_ref/SNAG_MMEA), as
tests/test_reference_e2e_gpu.py does for the default bf16 route:

  * test_main_py_train_precision_fp32: `python -m snag_b200.patch --train-precision fp32 <ref> ...` trains, evaluates and
    writes its prediction file like the stock run.
  * test_patched_fp32_forward_matches_reference: the same SNAG weights, noise state and dropout draws through the stock
    and the patched classes with loss.TRAIN_PRECISION = "fp32": SNAG.forward's loss within 1e-3 relative and the
    parameter gradients within 5e-3 (relative Frobenius) — against 5e-3 / 2e-2 for the bf16 route, whose rounded
    operands dominate those figures. The fp32 route's own error against fp64 is below 1e-5 relative in NLL
    (tests/test_loss_fp32_gpu.py); the rest of the margin covers the patched encoder and fusion kernels around it.
Skips without a reference checkout (baseline/install_ref.py)."""
from __future__ import annotations

import os
import re
import sys

import numpy as np
import pytest
import torch

from baseline import harness
from tests.test_reference_e2e_gpu import NUM, _metric_lines, _relerr, _run

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(harness.ref_root() is None, reason="no reference checkout (baseline/install_ref.py)")]


def test_main_py_train_precision_fp32(cuda_device, tmp_path):
    ref = harness.ref_root()
    n_side, n_links, epochs = 1500, 1000, 2
    data = tmp_path / "fp32"
    harness.write_dataset(str(data), n_side=n_side, n_links=n_links)
    out = _run([sys.executable, "-m", "snag_b200.patch", "--train-precision", "fp32", ref]
               + harness.main_argv(str(data), epochs=epochs, batch_size=256), cwd=ref)
    assert len(_metric_lines(out)) == 2 * (epochs + 1), out[-3000:]
    res = re.search(rf"Res:\[({NUM})\t({NUM})\t({NUM})\]", out)
    assert res and float(res[1]) > 0.2, out[-3000:]


def test_patched_fp32_forward_matches_reference(cuda_device, tmp_path, monkeypatch):
    from snag_b200 import loss as sloss, patch as spatch
    root = harness.load_reference()
    data = tmp_path / "data"
    harness.write_dataset(str(data), n_side=2000, n_links=1400, img_dim=512)
    cfgs = harness.parse_args(harness.main_argv(str(data), epochs=2, batch_size=400))
    cfgs.device = torch.device("cuda:0")
    cwd = os.getcwd()
    os.chdir(root)
    import importlib
    import logging
    import main as ref_main
    ref_snag = importlib.import_module("model.SNAG")
    logger = logging.getLogger("snag_e2e_fp32")
    logger.propagate = False
    monkeypatch.setattr(sloss, "TRAIN_PRECISION", "bf16")
    try:
        runner = ref_main.Runner(cfgs, None, logger)
        model = runner.model
        batch = np.asarray(runner.train_ill[:400], dtype=np.int32)
        torch.manual_seed(7)
        model.train()
        model.update_noise()
        noise_state = {k: getattr(model, k).clone() for k in ("rel_noisy_features", "att_noisy_features",
                                                              "img_noisy_features", "entity_noise", "entity_noise_mask")}
        model.zero_grad(set_to_none=True)
        torch.manual_seed(11)
        loss_ref, _ = model(batch)
        loss_ref.backward()
        grads_ref = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}

        spatch.patch(ref_main, train_precision="fp32")
        assert sloss.TRAIN_PRECISION == "fp32"
        torch.manual_seed(7)
        model_p = ref_snag.SNAG(runner.KGs, cfgs).cuda()
        model_p.load_state_dict(model.state_dict(), strict=True)
        model_p.train()
        for k, v in noise_state.items():
            setattr(model_p, k, v.clone())
        model_p.zero_grad(set_to_none=True)
        torch.manual_seed(11)
        loss_p, _ = model_p(batch)
        loss_p.backward()
        grads_p = {n: p.grad.detach().clone() for n, p in model_p.named_parameters() if p.grad is not None}
        rel_loss = abs(loss_p.item() - loss_ref.item()) / abs(loss_ref.item())
        flat_p = torch.cat([grads_p[n].reshape(-1) for n in sorted(grads_ref)])
        flat_r = torch.cat([grads_ref[n].reshape(-1) for n in sorted(grads_ref)])
        print(f"fp32 training route vs stock SNAG.forward: loss rel {rel_loss:.3g}, gradients rel {_relerr(flat_p, flat_r):.3g}")
        assert rel_loss <= 1e-3, (loss_p.item(), loss_ref.item())
        assert set(grads_p) == set(grads_ref)
        assert _relerr(flat_p, flat_r) < 5e-3, _relerr(flat_p, flat_r)
    finally:
        spatch.unpatch()
        os.chdir(cwd)
