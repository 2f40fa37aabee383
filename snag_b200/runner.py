"""Runner._test — host-side mirror of the reference's evaluation method (SNAG_MMEA/main.py:359-455), installed
on the reference's Runner class by snag_b200.patch. Same signature, same log lines (same rounding and format
strings), same prediction CSV, same side effects on the runner (early-stop counter, loss_log, best weights);
the N x N distance matrix, the CSLS temporaries and the 2n per-row torch.sort + .item() loops are replaced by
the fused sweeps of snag_b200.evaluate."""
from __future__ import annotations

import copy
import csv
import gc
import os
import os.path as osp

import numpy as np
import torch
import torch.nn.functional as F

from . import evaluate


def _test(self, test_left, test_right, last_epoch=False, save_name="", loss=None):
    with torch.no_grad():
        if self.args.model_name in ["EVA", "MCLEA"]:                                      # main.py:361-372
            if self.args.model_name == "EVA":
                self.model.emb_generat()
                w_normalized = F.softmax(self.model.weight_raw, dim=0)
            else:
                w_normalized = F.softmax(self.model.multimodal_encoder.fusion.weight.reshape(-1), dim=0)
            appdx = ""
            if self.args.w_name and self.args.w_char:
                appdx = f"-[name_{w_normalized[4]:.3f}]-[char_{w_normalized[5]:.3f}]"
            self.logger.info(f"weight_raw:[img_{w_normalized[0]:.3f}]-[attr_{w_normalized[1]:.3f}]-[rel_{w_normalized[2]:.3f}]-[graph_{w_normalized[3]:.3f}]{appdx}")
        if self.args.model_name in ["SNAG"]:                                              # main.py:374-378
            final_emb, weight_norm = self.model.joint_emb_generat()
        else:
            final_emb = self.model.joint_emb_generat()
        if self.args.distance == 1:
            # main.py:387-390: cityblock distances (scipy on the host in the reference) — materialised on the device
            out = evaluate.evaluate_alignment_l1(final_emb.float().contiguous(), test_left, test_right,
                                                 csls=self.args.csls is True, csls_k=self.args.csls_k,
                                                 want_top3=bool(last_epoch))
        else:
            # F.normalize (main.py:379), the gathers final_emb[test_left/right] (:386), pairwise_distances, csls_sim (:393)
            # and both ranking loops (:400-429) in one call; the normalisation happens on the gathered rows only
            out = evaluate.evaluate_alignment(final_emb.float().contiguous(), test_left, test_right,
                                              csls=self.args.csls is True, csls_k=self.args.csls_k,
                                              want_top3=bool(last_epoch), precision=evaluate.EVAL_PRECISION)
    top_k = [1, 10, 50]
    l2r, r2l = out["l2r"], out["r2l"]
    acc_l2r, mean_l2r, mrr_l2r = l2r.acc, l2r.mr, l2r.mrr
    acc_r2l, mean_r2l, mrr_r2l = r2l.acc, r2l.mr, r2l.mrr

    if last_epoch:                                                                        # main.py:395-420
        ranks = out["ranks"].rank_l2r.cpu().numpy()
        top3 = out["ranks"].top3_idx.cpu().numpy()
        test_left_np = test_left.cpu().numpy()
        test_right_np = test_right.cpu().numpy()
        to_write = [["idx", "rank", "query_id", "gt_id", "ret1", "ret2", "ret3"]]
        n_ret = min(3, test_right_np.shape[0])
        for idx in range(test_left_np.shape[0]):
            rets = [test_right_np[top3[idx, t]] for t in range(n_ret)]
            to_write.append([idx, int(ranks[idx]), test_left_np[idx], test_right_np[idx], *rets])
        if save_name == "":
            save_name = self.args.model_name
        save_pred_path = osp.join(self.args.data_path, self.args.model_name, f"{save_name}_pred")
        os.makedirs(save_pred_path, exist_ok=True)
        with open(osp.join(save_pred_path, f"{self.args.data_choice}_pred.txt"), "w") as f:
            wr = csv.writer(f, dialect='excel')
            wr.writerows(to_write)
    gc.collect()

    Loss_out = f", Loss = {self.loss_item:.4f}"                                          # main.py:439-444
    self.logger.info(f"Ep {self.epoch} | l2r: acc of top {top_k} = {acc_l2r}, mr = {mean_l2r:.3f}, mrr = {mrr_l2r:.3f}{Loss_out}")
    self.logger.info(f"Ep {self.epoch} | r2l: acc of top {top_k} = {acc_r2l}, mr = {mean_r2l:.3f}, mrr = {mrr_r2l:.3f}{Loss_out}")
    if last_epoch:
        t1, t2, t3 = acc_l2r
        self.logger.info(f"Res:[{t1}\t{t2}\t{mrr_l2r:.3f}]")

    self.early_stop_count -= 1                                                            # main.py:447-455
    if mrr_l2r > max(self.loss_log.acc) and not last_epoch:
        self.logger.info(f"Best model update in Ep {self.epoch}: MRR from [{max(self.loss_log.acc)}] --> [{mrr_l2r}] ... ")
        self.loss_log.update_acc(mrr_l2r)
        self.early_stop_count = self.early_stop_init
        self.best_model_wts = copy.deepcopy(self.model.state_dict())
