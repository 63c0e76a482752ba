"""Evaluation on the engine: PaSCo's SSC, panoptic-quality and uncertainty metrics (the metric side of
Net.step_inference(eval=True), net_panoptic_sparse.py:581-765).

The per-cell and per-row work runs in three CUDA sweeps (csrc/eval.cu through ops.eval_ssc / eval_pairs / eval_calib):

  SSCMetrics.add_batch / add_batch_ece   metrics.py:480-547,618-690   one sweep over the K x cells probability volume:
                                          [K,K] confusion, calibration bins and Σ NLL split by empty / non-empty prediction
  pq_compute_single_core, find_matched_  panoptic_quality.py:96-261   (n_gt+1) x (n_pred+1) intersection table of the GT and
  segment                                                             predicted panoptic ids over known cells
  UncertaintyMetrics.compute_ece_panop   metrics.py:98-166            calibration bins of the per-voxel mask confidences

and each scene's tables come to the host in ONE device→host copy.  What is left is small-table bookkeeping (matching,
PQ, ECE from bins), plain Python / numpy on the host.  The reference computes the same from dense [256,256,32] volumes
on the host (np.where per class, np.unique over 2.1 M uint64 keys).

Calibration follows torchmetrics' binary_calibration_error with its default 15 bins: confidence = the prediction,
accuracy = the target, bin boundaries torch.linspace(0, 1, n_bins + 1) in fp32, slot = bucketize(conf, boundaries,
right=True) - 1 over n_bins + 1 slots, ECE = Σ |acc - conf| · count / Σ count (NaN when there is no sample).
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F

from . import ops
from ._lib import PascoError
from .ensemble import SCENE, ensemble_panop, ensemble_sem_compl, panoptic_inference

N_BINS = 15
THING_IDS = (1, 2, 3, 4, 5, 6, 7, 8)

CUDA_KERNELS = SimpleNamespace(eval_ssc=ops.eval_ssc, eval_pairs=ops.eval_pairs, eval_calib=ops.eval_calib)


def calibration_bounds(n_bins: int = N_BINS, device=None) -> torch.Tensor:
    return torch.linspace(0, 1, n_bins + 1, dtype=torch.float32, device=device)


def ece_from_bins(count, sum_conf, sum_correct) -> float:
    """torchmetrics' l1 calibration error from per-slot (count, Σ confidence, Σ correct); NaN for an empty set."""
    count = np.asarray(count, dtype=np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        conf = np.nan_to_num(np.asarray(sum_conf, dtype=np.float64) / count)
        acc = np.nan_to_num(np.asarray(sum_correct, dtype=np.float64) / count)
        return float(np.sum(np.abs(acc - conf) * (count / count.sum())))


def calibration_error(conf: torch.Tensor, correct: torch.Tensor, n_bins: int = N_BINS) -> float:
    """binary_calibration_error(conf, correct) on a small host-side set (instance confidences)."""
    conf = conf.detach().float().cpu().reshape(-1)
    slot = (torch.bucketize(conf, calibration_bounds(n_bins), right=True) - 1).numpy()
    nb = n_bins + 1
    return ece_from_bins(np.bincount(slot, minlength=nb), np.bincount(slot, conf.double().numpy(), minlength=nb),
                         np.bincount(slot, correct.detach().cpu().reshape(-1).double().numpy(), minlength=nb))


def gt_panoptic(labels: torch.Tensor, masks: torch.Tensor, thing_ids: Sequence[int]):
    """convert_mask_label_to_panoptic_output (panoptic_quality.py:357-390) with torch on the masks' device, no host
    round trip: masks bool [n, X, Y, Z] paint in order (later masks overwrite earlier ones, label-0 masks paint nothing);
    a thing mask or the first stuff mask of its class opens a new segment id, a later stuff mask of the same class
    paints the first one's id.  Returns (gt_id int32 [cells], seg int64 [n] = id painted by each mask (0 = none),
    opens bool [n], area int64 [n] = each mask's full sum (the area of the segment it opens, unknown cells included))."""
    dev = masks.device
    n = masks.shape[0]
    lab = labels.to(dev).long().view(-1)
    flat = masks.reshape(n, -1)
    idx = torch.arange(n, device=dev)
    nz = lab != 0
    thing = torch.isin(lab, torch.as_tensor(list(thing_ids), device=dev, dtype=torch.long))
    same_before = (lab[:, None] == lab[None, :]) & (idx[None, :] < idx[:, None]) & nz[None, :]
    repeat = same_before.any(1)
    opens = nz & (thing | ~repeat)
    new_id = torch.cumsum(opens.long(), 0)
    first = torch.where(repeat, same_before.int().argmax(1), idx)
    seg = torch.where(nz, torch.where(opens, new_id, new_id[first]), torch.zeros_like(new_id))
    gt_id = torch.zeros(flat.shape[1], dtype=torch.int32, device=dev)
    seg32 = seg.int()
    for i in range(n):
        gt_id = torch.where(flat[i] & nz[i], seg32[i], gt_id)
    return gt_id, seg, opens, flat.sum(1)


class Evaluator:
    """One accumulator per eval instance (subnet i or the ensemble), as the reference keeps one SSCMetrics, PQStat and
    UncertaintyMetrics per i_infer.  stats() returns the reference's keys and values:

      "ssc"          SSCMetrics.get_stats() without inference_time
      "pq"           PQStat.pq_average for "All" (with "per_class"), "Things" and "Stuff" (pq_dagger, pq, sq, rq, n)
      "uncertainty"  UncertaintyMetrics.get_stats() at the reference's matching threshold 0.5: mask_ece, ins_ece,
                     ins_nll, count.  The reference's AUPRC, AUROC and FPR95 are hard-coded 0 (metrics.py:168-177) and its
                     mask_nll and ins_brier are never accumulated, so they are left out.

    `kernels` supplies eval_ssc / eval_pairs / eval_calib with the signatures of the ops functions (default: the CUDA
    sweeps); the tests substitute a torch restatement to check the host logic without a device."""

    def __init__(self, n_classes: int = 20, thing_ids: Sequence[int] = THING_IDS, compute_uncertainty: bool = False,
                 n_bins: int = N_BINS, kernels=None):
        self.n_classes, self.thing_ids, self.n_bins = n_classes, tuple(int(t) for t in thing_ids), n_bins
        self.compute_uncertainty = compute_uncertainty
        self.kernels = kernels or CUDA_KERNELS
        self.reset()

    def reset(self):
        K = self.n_classes
        self.completion = np.zeros(3, dtype=np.int64)                    # tp, fp, fn
        self.tps, self.fps, self.fns = (np.zeros(K, dtype=np.int64) for _ in range(3))
        self.empty_ece = self.nonempty_ece = 0.0
        self.empty_nll = self.nonempty_nll = 0.0
        self.n_empty = self.n_nonempty = 0
        self.ece_count = 0
        self.pq_per_cat: Dict[int, Dict[str, float]] = {}
        self.ins_confs: List[float] = []
        self.ins_correct: List[bool] = []
        self.ins_probs: List[torch.Tensor] = []
        self.ins_labels: List[int] = []
        self.mask_bins: List[torch.Tensor] = []                         # per scene, on the device until stats()
        self.scene_count = 0

    def _cat(self, c: int) -> Dict[str, float]:
        return self.pq_per_cat.setdefault(int(c), {"all_iou": 0.0, "all_n": 0.0, "iou": 0.0, "tp": 0, "fp": 0, "fn": 0})

    @torch.no_grad()
    def add_scene(self, prob: torch.Tensor, pan: torch.Tensor, lin: torch.Tensor, vox_conf: Optional[torch.Tensor],
                  segments_info: List[Dict], semantic_label: torch.Tensor, mask_label: Dict) -> None:
        """prob float [K, X, Y, Z] (ensemble_sem_compl's volume); pan int32 [N] panoptic ids at cells lin [N] and vox_conf
        [N] (panoptic_inference(return_confidence=True)); segments_info its segment list; semantic_label_origin uint8
        [X, Y, Z] (255 = unknown); mask_label_origin {"labels": [n], "masks": bool [n, X, Y, Z]}."""
        K = prob.shape[0]
        dev = prob.device
        prob = prob.reshape(K, -1).float().contiguous()
        cells = prob.shape[1]
        label = semantic_label.to(dev).reshape(-1).to(torch.uint8).contiguous()
        gt_id, seg, opens, area = gt_panoptic(mask_label["labels"], mask_label["masks"].to(dev), self.thing_ids)
        n_gt = int(seg.shape[0])                                          # segment ids are at most the mask count
        n_pred = max((int(s["id"]) for s in segments_info), default=0)
        pan = pan.to(torch.int32).contiguous()
        lin = lin.to(torch.int64).contiguous()
        nb = self.n_bins + 1
        bounds = calibration_bounds(self.n_bins, dev)
        n_ssc = K * K + 4 * nb
        n_sum = 2 * nb + 2
        n_tab = (n_gt + 1) * (n_pred + 1)
        sizes = [n_ssc, n_sum, n_tab, n_gt, n_gt, n_gt, n_gt, 1]
        buf = torch.zeros(sum(sizes), dtype=torch.int64, device=dev)
        counts, sums, table, b_lab, b_seg, b_opens, b_area, b_err = torch.split(buf, sizes)
        self.kernels.eval_ssc(prob, label, bounds, counts, sums.view(torch.float64))
        self.kernels.eval_pairs(pan, lin, gt_id, label, n_gt, n_pred, table)
        b_lab.copy_(mask_label["labels"].to(dev).view(-1))
        b_seg.copy_(seg)
        b_opens.copy_(opens)
        b_area.copy_(area)
        err = ops._err_flag(dev) if dev.type == "cuda" else torch.zeros(1, dtype=torch.int32)
        b_err.copy_(err)
        host = buf.cpu().numpy()                                          # the one device→host copy of the scene
        h_counts, h_sums, h_table, h_lab, h_seg, h_opens, h_area, h_err = np.split(host, np.cumsum(sizes)[:-1])
        if int(h_err[0]) == ops.EVAL_ERR_ID:
            err.zero_()
            raise PascoError("evaluation: a label >= n_classes or a segment id beyond its table "
                             f"(GT ids <= {n_gt}, predicted ids <= {n_pred})")
        h_sums = h_sums.view(np.float64)
        self._add_ssc(h_counts.reshape(-1), h_sums, K)
        matched = self._add_panoptic(h_table.reshape(n_gt + 1, n_pred + 1), h_lab, h_seg, h_opens, h_area, segments_info)
        if self.compute_uncertainty:
            match = torch.zeros(n_pred + 1, dtype=torch.int32)
            for p, g in matched.items():
                match[p] = g
            out = torch.zeros(3 * nb, dtype=torch.int64, device=dev)
            self.kernels.eval_calib(vox_conf.float().contiguous(), pan, lin, gt_id, label, match.to(dev), bounds,
                                    out[:2 * nb], out[2 * nb:].view(torch.float64))
            self.mask_bins.append(out)
            self.scene_count += 1

    def _add_ssc(self, counts: np.ndarray, sums: np.ndarray, K: int) -> None:
        nb = self.n_bins + 1
        conf = counts[:K * K].reshape(K, K)                               # [target, prediction]
        tp = np.diag(conf)
        self.tps += tp
        self.fps += conf.sum(0) - tp
        self.fns += conf.sum(1) - tp
        self.completion += [conf[1:, 1:].sum(), conf[0, 1:].sum(), conf[1:, 0].sum()]
        if not self.compute_uncertainty:
            return
        cnt = counts[K * K:K * K + 2 * nb].reshape(2, nb)
        cor = counts[K * K + 2 * nb:K * K + 4 * nb].reshape(2, nb)
        sconf = sums[:2 * nb].reshape(2, nb)
        self.empty_ece += ece_from_bins(cnt[0], sconf[0], cor[0])
        self.nonempty_ece += ece_from_bins(cnt[1], sconf[1], cor[1])
        self.empty_nll += float(sums[2 * nb])
        self.nonempty_nll += float(sums[2 * nb + 1])
        self.n_empty += int(cnt[0].sum())
        self.n_nonempty += int(cnt[1].sum())
        self.ece_count += 1

    def _add_panoptic(self, table, lab, seg, opens, area, segments_info) -> Dict[int, int]:
        """pq_compute_single_core + find_matched_segment(threshold=0.5) on the intersection table, after the reference
        drops the segments that only lie in unknown cells (net_panoptic_sparse.py:724-732).  Returns pred id → GT id."""
        gt_present = table.sum(1) > 0
        pred_area = table.sum(0)
        gt_segms = {int(seg[i]): {"category_id": int(lab[i]), "area": int(area[i])}
                    for i in range(len(seg)) if opens[i] and gt_present[int(seg[i])]}
        pred_segms = {int(s["id"]): dict(s, area=int(pred_area[int(s["id"])]))
                      for s in segments_info if pred_area[int(s["id"])] > 0}
        gt_matched, pred_matched, matched = set(), set(), {}
        gs, ps = np.nonzero(table)
        for g, p in zip(gs.tolist(), ps.tolist()):                        # ascending (gt, pred), as np.unique orders them
            if g == 0 or p == 0 or g not in gt_segms or p not in pred_segms:
                continue
            inter = int(table[g, p])
            gi, pi = gt_segms[g], pred_segms[p]
            iou = inter / (pi["area"] + gi["area"] - inter)
            if iou > 0.5:
                matched[p] = g                                            # find_matched_segment: any category
            if gi["category_id"] != pi["category_id"]:
                continue
            if gi["category_id"] not in self.thing_ids:
                st = self._cat(gi["category_id"])
                st["all_iou"] += iou
                st["all_n"] += 1
                pred_matched.add(p)
            if iou > 0.5:
                st = self._cat(gi["category_id"])
                st["tp"] += 1
                st["iou"] += iou
                gt_matched.add(g)
                pred_matched.add(p)
        for g, gi in gt_segms.items():
            if g not in gt_matched:
                self._cat(gi["category_id"])["fn"] += 1
        for p, pi in pred_segms.items():
            if p not in pred_matched:
                self._cat(pi["category_id"])["fp"] += 1
        if self.compute_uncertainty:
            for p, pi in pred_segms.items():                              # compute_ece_panop's instance terms
                self.ins_confs.append(float(pi["confidence"]))
                self.ins_probs.append(pi["all_class_probs"])
                g = matched.get(p)
                if g is None:
                    self.ins_correct.append(False)
                    self.ins_labels.append(self.n_classes)
                else:
                    self.ins_correct.append(gt_segms[g]["category_id"] == pi["category_id"])
                    self.ins_labels.append(gt_segms[g]["category_id"])
        return matched

    def pq_average(self, isthing: Optional[bool]):
        """PQStat.pq_average(isthing, ignore_cat_id=0, thing_ids) (panoptic_quality.py:49-93)."""
        pq_dagger = pq = sq = rq = 0.0
        n = 0
        per_class = {}
        for label, s in self.pq_per_cat.items():
            if label == 0:
                continue
            if isthing is not None and isthing != (label in self.thing_ids):
                continue
            tp, fp, fn = s["tp"], s["fp"], s["fn"]
            if tp + fp + fn == 0:
                per_class[label] = {"pq": 0.0, "sq": 0.0, "rq": 0.0}
                continue
            n += 1
            pq_c = s["iou"] / (tp + 0.5 * fp + 0.5 * fn)
            sq_c = s["iou"] / tp if tp != 0 else 0
            rq_c = tp / (tp + 0.5 * fp + 0.5 * fn)
            per_class[label] = {"pq": pq_c, "sq": sq_c, "rq": rq_c}
            pq, sq, rq = pq + pq_c, sq + sq_c, rq + rq_c
            if isthing is None:
                pq_dagger += pq_c if label in self.thing_ids else s["all_iou"] / max(s["all_n"], 1)
        n = max(n, 1)
        return {"pq_dagger": pq_dagger / n, "pq": pq / n, "sq": sq / n, "rq": rq / n, "n": n}, per_class

    def stats(self) -> Dict:
        tp, fp, fn = (int(v) for v in self.completion)
        if tp != 0:
            precision, recall, iou = tp / (tp + fp), tp / (tp + fn), tp / (tp + fp + fn)
        else:
            precision = recall = iou = 0
        iou_ssc = self.tps / (self.tps + self.fps + self.fns + 1e-5)
        c = self.ece_count
        ssc = {"precision": precision, "recall": recall, "iou": iou, "iou_ssc": iou_ssc,
               "iou_ssc_mean": np.mean(iou_ssc[1:]),
               "empty_ece": self.empty_ece / c if c else 0, "nonempty_ece": self.nonempty_ece / c if c else 0,
               "empty_nll": self.empty_nll / self.n_empty if self.n_empty else 0,
               "nonempty_nll": self.nonempty_nll / self.n_nonempty if self.n_nonempty else 0}
        pq = {}
        for name, isthing in (("All", None), ("Things", True), ("Stuff", False)):
            pq[name], per_class = self.pq_average(isthing)
            if name == "All":
                pq["per_class"] = per_class
        out = {"ssc": ssc, "pq": pq}
        if self.compute_uncertainty:
            out["uncertainty"] = self._uncertainty_stats()
        return out

    def _uncertainty_stats(self) -> Dict:
        nb = self.n_bins + 1
        mask_ece = 0.0
        if self.mask_bins:
            bins = torch.stack(self.mask_bins).cpu()
            for b in bins:
                cnt, cor, sconf = b[:nb].numpy(), b[nb:2 * nb].numpy(), b[2 * nb:].view(torch.float64).numpy()
                mask_ece += ece_from_bins(cnt, sconf, cor) if cnt.sum() else 0.0   # no valid voxel adds 0
            mask_ece /= self.scene_count
        if self.ins_probs:
            probs = torch.stack(self.ins_probs, 0)
            labels = torch.as_tensor(self.ins_labels, device=probs.device)
            ins_nll = F.nll_loss(torch.log(probs + 1e-8), labels, reduction="mean").item()
        else:
            ins_nll = 0.0
        ins_ece = calibration_error(torch.tensor(self.ins_confs), torch.tensor(self.ins_correct), self.n_bins) \
            if self.ins_confs else 0
        return {"mask_ece": mask_ece, "ins_ece": ins_ece, "ins_nll": ins_nll, "count": len(self.ins_confs)}


def evaluate_step(net, batch: Dict, step_type: str, evaluators: Sequence[Evaluator], overlap_threshold: float = 0.4,
                  object_mask_threshold: float = 0.7, iou_threshold: float = 0.2, thing_ids: Sequence[int] = THING_IDS,
                  size=SCENE):
    """Net.step_inference(eval=True) (net_panoptic_sparse.py:546-648) on the engine for one scene: PascoNet forward,
    ensembling, panoptic inference with confidences, then Evaluator.add_scene for subnet 0 and the ensemble ("val") or
    every subnet and the ensemble ("test").  evaluators[i] accumulates eval instance i (M + 1 of them).  The batch holds
    the network inputs (as synthetic.make_scene builds them, on the device), "semantic_label_origin" [1, X, Y, Z] and
    "mask_label_origin" [{"labels", "masks"}].  Returns the panoptic outputs (pan, lin, vox_conf, segments_info)."""
    with torch.no_grad():
        out = net(batch["in_feats"], batch["in_coords"], batch["global_min_Cs"], batch["global_max_Cs"], batch["min_Cs"],
                  batch["max_Cs"], test=step_type == "test")
        Ts = batch["Ts"]
        sem = [(t.F, t.C[:, 1:]) for t in out["sem_logits_pruneds"]]
        sem_d = ensemble_sem_compl(sem, Ts, size)
        preds = [{"voxel_logits": (p["voxel_logits"].F, p["voxel_logits"].C[:, 1:]), "query_logits": p["query_logits"]}
                 for p in out["panop_predictions"]]
        ens = ensemble_panop(preds, sem_d, Ts, iou_threshold=iou_threshold, size=size)
        eval_list = [0, len(ens) - 1] if step_type == "val" else range(len(ens))
        outs = []
        for i in eval_list:
            prob, lin = ens[i]["voxel_probs"]
            pan, _, infos, conf = panoptic_inference(prob, ens[i]["query_probs"][0], overlap_threshold,
                                                     object_mask_threshold, thing_ids, return_confidence=True)
            evaluators[i].add_scene(sem_d[i], pan, lin, conf, infos, batch["semantic_label_origin"][0],
                                    batch["mask_label_origin"][0])
            outs.append((pan, lin, conf, infos))
        return outs
