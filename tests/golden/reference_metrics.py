"""Runs the reference's OWN metric code (Net.evaluate_all, net_panoptic_sparse.py:650-765, with SSCMetrics, PQStat and
UncertaintyMetrics from pasco/models/metrics.py and pasco/loss/panoptic_quality.py) on given outputs, from an upstream
package root (oracle/_ref as build() compiles it, or a checkout).  Used by tests/test_evaluation.py and
tools/eval_bench.py to compare the engine's evaluator with the reference on the same outputs.

binary_calibration_error is the restatement of torchmetrics' definition in metrics_scenes.py (torchmetrics is not
installed; the compat stub bins differently below 0.5)."""
import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


class ReferenceMetrics:
    def __init__(self, ref_root, n_instances, n_classes=20, thing_ids=(1, 2, 3, 4, 5, 6, 7, 8)):
        for p in (HERE, ref_root, os.path.join(ROOT, "compat")):
            if p not in sys.path:
                sys.path.insert(0, p)
        import metrics_scenes
        import pasco.models.metrics as RM
        from pasco.loss.panoptic_quality import PQStat
        from pasco.models.net_panoptic_sparse import Net
        RM.binary_calibration_error = metrics_scenes.binary_calibration_error
        self.Net, self.thing_ids = Net, list(thing_ids)
        self.ssc = [RM.SSCMetrics(n_classes) for _ in range(n_instances)]
        self.pq = [PQStat() for _ in range(n_instances)]
        self.unc = [RM.UncertaintyMetrics() for _ in range(n_instances)]
        self.net = types.SimpleNamespace(thing_ids=self.thing_ids, n_classes=n_classes, uncertainty_thresholds=[0.5],
                                         uncertainty_metrics_by_thresholds={0.5: self.unc})
        self.net.evaluate_panoptic = types.MethodType(Net.evaluate_panoptic, self.net)

    def add_scene(self, i, prob, pan, lin, vox_conf, segments_info, semantic_label, mask_label):
        """Densifies the sparse panoptic output onto the grid as helper.panoptic_inference returns it, then
        evaluate_all in test mode (compute_uncertainty=True).  mask_label stays on the host as the reference needs."""
        size = prob.shape[1:]
        dev = prob.device
        pan_d = torch.zeros(prob[0].numel(), dtype=torch.int32, device=dev)
        pan_d[lin] = pan.to(torch.int32)
        conf_d = torch.zeros(prob[0].numel(), dtype=torch.float32, device=dev)
        conf_d[lin] = vox_conf.float()
        out = {"panoptic_seg_denses": pan_d.view(1, *size), "segments_infos": [segments_info],
               "vox_confidence_denses": conf_d.view(1, *size), "vox_all_mask_probs_denses": [None]}
        label = semantic_label.to(dev).long().unsqueeze(0)
        self.Net.evaluate_all(self.net, ssc_confidence=prob.max(0)[0], i_infer=i, sem_prob=prob, panop_out=out,
                              semantic_label=label, mask_labels=[{"labels": mask_label["labels"].cpu(),
                                                                  "masks": mask_label["masks"].cpu()}],
                              ssc_metrics=self.ssc[i], pq_stat=self.pq[i], uncertainty_metrics=self.unc[i],
                              compute_uncertainty=True)

    def stats(self, i):
        s = self.ssc[i].get_stats()
        s.pop("inference_time")
        pq = {}
        for name, isthing in (("All", None), ("Things", True), ("Stuff", False)):
            pq[name], per_class = self.pq[i].pq_average(isthing=isthing, ignore_cat_id=0, thing_ids=self.thing_ids)
            if name == "All":
                pq["per_class"] = per_class
        u = self.unc[i].get_stats()
        return {"ssc": s, "pq": pq, "uncertainty": {k: u[k] for k in ("mask_ece", "ins_ece", "ins_nll", "count")}}
