"""Golden vectors for pasco_b200/evaluation.py: runs the reference's OWN metric code from an upstream PaSCo checkout
(PASCO_REFERENCE, default oracle/build_ref.DEFAULT_CHECKOUT) on the CPU (MinkowskiEngine = the oracle shim) over the
seeded scenes of metrics_scenes.py:
helper.panoptic_inference, then Net.evaluate_all (net_panoptic_sparse.py:650-765: SSCMetrics.add_batch / add_batch_ece,
convert_mask_label_to_panoptic_output, pq_compute_single_core, find_matched_segment, UncertaintyMetrics.compute_ece_panop),
and at the end SSCMetrics.get_stats, PQStat.pq_average and UncertaintyMetrics.get_stats per eval instance.

    python tests/golden/make_golden_metrics.py

Patches, in this process only:
  - torchmetrics is not installed; the compat stub's binary_calibration_error folds p < 0.5 to 1 - p, torchmetrics does
    not.  metrics.binary_calibration_error is replaced by metrics_scenes.binary_calibration_error, the restatement of
    torchmetrics' definition; each call's bins are recorded for the table checks.
  - UncertaintyMetrics.get_stats calls Tensor.cuda(); it is made the identity (the generator runs on the CPU).
"""
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [os.path.join(ROOT, "oracle"), HERE]
from build_ref import DEFAULT_CHECKOUT  # noqa: E402
sys.path[:0] = [os.path.join(ROOT, "oracle", "shims"), os.path.join(ROOT, "compat"),
                os.environ.get("PASCO_REFERENCE") or DEFAULT_CHECKOUT, ROOT]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import metrics_scenes as S  # noqa: E402

SEEDS = (0, 1)
OVERLAP, OBJECT_MASK = 0.4, 0.5
OFFSET = 256 * 256 * 256


def main():
    import MinkowskiEngine as ME
    import pasco.models.metrics as RM
    from pasco.models.helper import panoptic_inference
    from pasco.models.net_panoptic_sparse import Net
    from pasco.loss.panoptic_quality import PQStat, convert_mask_label_to_panoptic_output

    record = []

    def recorded_bce(preds, target, n_bins=15, norm="l1", **kw):
        record.append([t.numpy() for t in S.calibration_bins(preds, target, n_bins)])
        return S.binary_calibration_error(preds, target, n_bins, norm)

    RM.binary_calibration_error = recorded_bce
    torch.Tensor.cuda = lambda self, *a, **k: self

    n = S.N_INSTANCES
    ssc = [RM.SSCMetrics(S.K) for _ in range(n)]
    pqs = [PQStat() for _ in range(n)]
    unc = [RM.UncertaintyMetrics() for _ in range(n)]
    net = types.SimpleNamespace(thing_ids=S.THING_IDS, n_classes=S.K, uncertainty_thresholds=[0.5],
                                uncertainty_metrics_by_thresholds={0.5: unc})
    net.evaluate_panoptic = types.MethodType(Net.evaluate_panoptic, net)
    scenes = [S.make_scene(s) for s in SEEDS]
    arrays = {"checksum": np.frombuffer(S.checksum(scenes).encode(), dtype=np.uint8)}
    for si, sc in enumerate(scenes):
        label = sc["semantic_label"].long().unsqueeze(0)
        gt_pan, _ = convert_mask_label_to_panoptic_output(sc["mask_label"]["labels"], sc["mask_label"]["masks"], S.THING_IDS)
        gt_pan = gt_pan.numpy().reshape(-1).copy()
        gt_pan[label.view(-1).numpy() == 255] = 0
        for i, ins in enumerate(sc["instances"]):
            lin = ins["lin"]
            X, Y, Z = S.GRID
            C = torch.stack([torch.zeros_like(lin), lin // (Y * Z), (lin // Z) % Y, lin % Z], 1).int()
            vp = ME.SparseTensor(ins["vox_probs"], C)
            out = panoptic_inference(vp, ins["query_probs"].unsqueeze(0), overlap_threshold=OVERLAP,
                                     object_mask_threshold=OBJECT_MASK, thing_ids=S.THING_IDS, min_C=torch.tensor([0, 0, 0]),
                                     scene_size=S.GRID, input_query_logit=False, input_voxel_logit=False)
            key = f"s{si}_i{i}"
            order = torch.argsort(vp.C[:, 1:].long() @ torch.tensor([Y * Z, Z, 1]))
            rows_lin = (vp.C[:, 1:].long() @ torch.tensor([Y * Z, Z, 1]))[order]
            assert torch.equal(rows_lin, lin)
            cc = vp.C[order].long()
            arrays[f"{key}_pan"] = out["panoptic_seg_denses"][0][cc[:, 1], cc[:, 2], cc[:, 3]].numpy()
            arrays[f"{key}_vox_conf"] = out["vox_confidence_denses"][0][cc[:, 1], cc[:, 2], cc[:, 3]].numpy()
            infos = out["segments_infos"][0]
            arrays[f"{key}_segments"] = np.array([[s["id"], int(s["isthing"]), s["category_id"], s["query_id"]] for s in infos]).reshape(-1, 4)
            arrays[f"{key}_all_class_probs"] = np.stack([s["all_class_probs"].numpy() for s in infos]).reshape(-1, S.K + 1)
            arrays[f"{key}_confidence"] = np.array([s["confidence"] for s in infos], dtype=np.float64)
            # intersections over known cells, as pq_compute_single_core counts them (np.unique of gt * OFFSET + pred)
            pred_pan = out["panoptic_seg_denses"][0].numpy().reshape(-1).copy()
            pred_pan[label.view(-1).numpy() == 255] = 0
            keys, cnt = np.unique(gt_pan.astype(np.uint64) * OFFSET + pred_pan.astype(np.uint64), return_counts=True)
            arrays[f"{key}_pairs"] = np.stack([keys // OFFSET, keys % OFFSET, cnt], 1).astype(np.int64)
            before = dict(tps=ssc[i].tps.copy(), fps=ssc[i].fps.copy(), fns=ssc[i].fns.copy(),
                          comp=np.array([ssc[i].completion_tp, ssc[i].completion_fp, ssc[i].completion_fn]),
                          nll=np.array([ssc[i].empty_nll, ssc[i].nonempty_nll, ssc[i].n_empty_voxels, ssc[i].n_nonempty_voxels]))
            n_rec = len(record)
            prob = ins["prob"]
            Net.evaluate_all(net, ssc_confidence=prob.max(0)[0], i_infer=i, sem_prob=prob, panop_out=out,
                             semantic_label=label, mask_labels=[sc["mask_label"]], ssc_metrics=ssc[i], pq_stat=pqs[i],
                             uncertainty_metrics=unc[i], compute_uncertainty=True)
            arrays[f"{key}_tps_fps_fns"] = np.stack([ssc[i].tps - before["tps"], ssc[i].fps - before["fps"], ssc[i].fns - before["fns"]])
            arrays[f"{key}_completion"] = np.array([ssc[i].completion_tp, ssc[i].completion_fp, ssc[i].completion_fn]) - before["comp"]
            arrays[f"{key}_nll"] = np.array([ssc[i].empty_nll, ssc[i].nonempty_nll, ssc[i].n_empty_voxels,
                                             ssc[i].n_nonempty_voxels]) - before["nll"]
            new = record[n_rec:]
            assert len(new) in (2, 3), len(new)
            arrays[f"{key}_ssc_bins"] = np.stack([np.stack(b) for b in new[-2:]])        # [empty/nonempty, 3, NB]
            arrays[f"{key}_mask_bins"] = np.stack(new[0]) if len(new) == 3 else np.zeros((3, 16))
    for i in range(n):
        st = ssc[i].get_stats()
        arrays[f"stats{i}_ssc"] = np.array([st[k] for k in ("precision", "recall", "iou", "iou_ssc_mean", "empty_ece",
                                                              "nonempty_ece", "empty_nll", "nonempty_nll")], dtype=np.float64)
        arrays[f"stats{i}_iou_ssc"] = np.asarray(st["iou_ssc"], dtype=np.float64)
        rows = []
        for name, isthing in (("All", None), ("Things", True), ("Stuff", False)):
            r, per_class = pqs[i].pq_average(isthing=isthing, ignore_cat_id=0, thing_ids=S.THING_IDS)
            rows.append([float(r[k]) for k in ("pq_dagger", "pq", "sq", "rq", "n")])
            if name == "All":
                arrays[f"stats{i}_per_class"] = np.array([[c, float(v["pq"]), float(v["sq"]), float(v["rq"])]
                                                          for c, v in per_class.items()], dtype=np.float64)
        arrays[f"stats{i}_pq"] = np.array(rows, dtype=np.float64)
        u = unc[i].get_stats()
        arrays[f"stats{i}_unc"] = np.array([float(u[k]) for k in ("mask_ece", "ins_ece", "ins_nll", "count")], dtype=np.float64)
    np.savez_compressed(os.path.join(HERE, "metrics_m3.npz"), **arrays)
    for i in range(n):
        print(i, arrays[f"stats{i}_ssc"], arrays[f"stats{i}_pq"][0], arrays[f"stats{i}_unc"])


if __name__ == "__main__":
    torch.set_num_threads(os.cpu_count())
    main()
