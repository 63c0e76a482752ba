"""pasco_b200/evaluation.py and the eval sweeps of csrc/eval.cu against the reference's own metric code.

The fixture (tests/golden/make_golden_metrics.py → metrics_m3.npz) holds what the reference's panoptic_inference,
Net.evaluate_all and the get_stats / pq_average calls computed on the CPU over two seeded 64 x 64 x 16 scenes with four
eval instances each (tests/golden/metrics_scenes.py).  The CPU tests run the host logic with a torch restatement of the
three sweeps; the GPU tests run the CUDA sweeps."""
import math
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(HERE, "golden"))
import metrics_scenes as S  # noqa: E402

G = np.load(os.path.join(HERE, "golden", "metrics_m3.npz"))
SEEDS = (0, 1)
OVERLAP, OBJECT_MASK = 0.4, 0.5
REF = os.environ.get("PASCO_REFERENCE") or os.path.join(ROOT, "oracle", "_ref")
NB = 16


def _scenes():
    sc = [S.make_scene(s) for s in SEEDS]
    assert S.checksum(sc) == G["checksum"].tobytes().decode(), "metrics_scenes.py no longer makes the fixture's inputs"
    return sc


# ---- torch restatement of the three sweeps (same outputs as ops.eval_ssc / eval_pairs / eval_calib) -----------------
def _t_ssc(prob, label, bounds, counts, sums):
    K = prob.shape[0]
    conf, pred = prob.max(0)
    lab = label.long()
    known = lab != 255
    t = torch.where(known, lab, 0)
    counts[:K * K] += torch.bincount((t * K + pred)[known], minlength=K * K)
    slot = torch.bucketize(conf, bounds, right=True) - 1 + NB * (pred != 0).long()
    counts[K * K:K * K + 2 * NB] += torch.bincount(slot[known], minlength=2 * NB)
    counts[K * K + 2 * NB:] += torch.bincount(slot[known & (pred == lab)], minlength=2 * NB)
    sums[:2 * NB] += torch.bincount(slot[known], conf[known].double(), minlength=2 * NB)
    nll = -torch.log(prob.gather(0, t.view(1, -1)).view(-1) + 1e-12)
    sums[2 * NB:] += torch.bincount((pred != 0).long()[known], nll[known].double(), minlength=2)


def _t_pairs(pred_id, row_cell, gt_id, label, n_gt, n_pred, table):
    pan = torch.zeros(gt_id.numel(), dtype=torch.long)
    pan[row_cell] = pred_id.long()
    known = label != 255
    table += torch.bincount(gt_id[known].long() * (n_pred + 1) + pan[known], minlength=(n_gt + 1) * (n_pred + 1))


def _t_calib(conf, pred_id, row_cell, gt_id, label, match, bounds, counts, sums):
    g = gt_id[row_cell].long()
    valid = (label[row_cell] != 255) & (g != 0) & (conf != 0)
    correct = match[pred_id.long()].long() == g
    slot = torch.bucketize(conf, bounds, right=True) - 1
    counts[:NB] += torch.bincount(slot[valid], minlength=NB)
    counts[NB:] += torch.bincount(slot[valid & correct], minlength=NB)
    sums += torch.bincount(slot[valid], conf[valid].double(), minlength=NB)


TORCH_KERNELS = SimpleNamespace(eval_ssc=_t_ssc, eval_pairs=_t_pairs, eval_calib=_t_calib)


class _Recorder:
    """Wraps a kernel set and keeps a host copy of every output table."""

    def __init__(self, k):
        self.k, self.log = k, []

    def _wrap(self, name, outs):
        def f(*a):
            getattr(self.k, name)(*a)
            self.log.append((name, [a[i].cpu().clone() for i in outs]))
        return f

    def __getattr__(self, name):
        return self._wrap(name, {"eval_ssc": (3, 4), "eval_pairs": (6,), "eval_calib": (7, 8)}[name])


def _run(dev, kernels):
    from pasco_b200 import ensemble as E
    from pasco_b200.evaluation import Evaluator
    rec = _Recorder(kernels)
    evs = [Evaluator(S.K, S.THING_IDS, compute_uncertainty=True, kernels=rec) for _ in range(S.N_INSTANCES)]
    for sc in _scenes():
        for i, ins in enumerate(sc["instances"]):
            pan, _, infos, conf = E.panoptic_inference(ins["vox_probs"].to(dev), ins["query_probs"].to(dev), OVERLAP,
                                                       OBJECT_MASK, S.THING_IDS, return_confidence=True)
            ml = {"labels": sc["mask_label"]["labels"].to(dev), "masks": sc["mask_label"]["masks"].to(dev)}
            evs[i].add_scene(ins["prob"].to(dev), pan, ins["lin"].to(dev), conf, infos, sc["semantic_label"].to(dev), ml)
    return evs, rec.log


def _close(a, b, tol, what):
    a, b = float(a), float(b)
    assert (math.isnan(a) and math.isnan(b)) or abs(a - b) <= tol * max(1.0, abs(b)), f"{what}: {a} vs {b}"


def _check_stats(st, i, tol=1e-5):
    ref = G[f"stats{i}_ssc"]
    for j, k in enumerate(("precision", "recall", "iou", "iou_ssc_mean", "empty_ece", "nonempty_ece", "empty_nll",
                           "nonempty_nll")):
        _close(st["ssc"][k], ref[j], tol, f"instance {i} {k}")
    assert np.allclose(st["ssc"]["iou_ssc"], G[f"stats{i}_iou_ssc"], rtol=0, atol=tol)
    for r, name in enumerate(("All", "Things", "Stuff")):
        for j, k in enumerate(("pq_dagger", "pq", "sq", "rq", "n")):
            _close(st["pq"][name][k], G[f"stats{i}_pq"][r, j], tol, f"instance {i} {name} {k}")
    pc = G[f"stats{i}_per_class"]
    assert [int(c) for c in pc[:, 0]] == list(st["pq"]["per_class"].keys())
    for c, pq, sq, rq in pc:
        got = st["pq"]["per_class"][int(c)]
        for k, v in (("pq", pq), ("sq", sq), ("rq", rq)):
            _close(got[k], v, tol, f"instance {i} class {int(c)} {k}")
    for j, k in enumerate(("mask_ece", "ins_ece", "ins_nll", "count")):
        _close(st["uncertainty"][k], G[f"stats{i}_unc"][j], tol, f"instance {i} {k}")


def _check_tables(log, rel=1e-6):
    K = S.K
    steps = iter(log)
    for si in range(len(SEEDS)):
        for i in range(S.N_INSTANCES):
            key = f"s{si}_i{i}"
            _, (counts, sums) = next(steps)
            _, (table,) = next(steps)
            _, (ccounts, csums) = next(steps)
            conf = counts[:K * K].view(K, K).numpy()
            tp = np.diag(conf)
            assert np.array_equal(np.stack([tp, conf.sum(0) - tp, conf.sum(1) - tp]), G[f"{key}_tps_fps_fns"]), key
            assert [conf[1:, 1:].sum(), conf[0, 1:].sum(), conf[1:, 0].sum()] == G[f"{key}_completion"].tolist(), key
            cnt = counts[K * K:K * K + 2 * NB].view(2, NB).numpy()
            cor = counts[K * K + 2 * NB:].view(2, NB).numpy()
            sf = sums.view(torch.float64).numpy()
            ref = G[f"{key}_ssc_bins"]                                         # [split, (count, Σconf, Σacc), slot]
            assert np.array_equal(cnt, ref[:, 0]) and np.array_equal(cor, ref[:, 2]), key
            assert np.allclose(sf[:2 * NB].reshape(2, NB), ref[:, 1], rtol=rel, atol=0), key
            nll = G[f"{key}_nll"]
            assert np.allclose(sf[2 * NB:], nll[:2], rtol=rel, atol=0) and cnt.sum(1).tolist() == nll[2:].tolist(), key
            pairs = G[f"{key}_pairs"]
            W = int(G[f"{key}_segments"][:, 0].max()) + 1 if len(G[f"{key}_segments"]) else 1   # n_pred + 1
            t = table.numpy().reshape(-1, W)
            for g, p, c in pairs:
                if g == 0 and p == 0:
                    continue                                                  # the reference counts unknown cells here
                assert t[g, p] == c, (key, g, p)
            nz = np.argwhere(t)
            assert {(g, p) for g, p in nz if (g, p) != (0, 0)} == {(g, p) for g, p, _ in pairs if (g, p) != (0, 0)}, key
            mb = G[f"{key}_mask_bins"]
            if mb[0].sum():
                assert np.array_equal(ccounts[:NB].numpy(), mb[0]) and np.array_equal(ccounts[NB:].numpy(), mb[2]), key
                assert np.allclose(csums.view(torch.float64).numpy(), mb[1], rtol=rel, atol=0), key


def test_panoptic_inference_confidences_match_the_reference():
    from pasco_b200 import ensemble as E
    for si, sc in enumerate(_scenes()):
        for i, ins in enumerate(sc["instances"]):
            key = f"s{si}_i{i}"
            pan, sem, infos, conf = E.panoptic_inference(ins["vox_probs"], ins["query_probs"], OVERLAP, OBJECT_MASK,
                                                         S.THING_IDS, return_confidence=True)
            assert np.array_equal(pan.numpy(), G[f"{key}_pan"]), key
            assert np.allclose(conf.numpy(), G[f"{key}_vox_conf"], rtol=0, atol=1e-7), key
            got = np.array([[s["id"], int(s["isthing"]), s["category_id"], s["query_id"]] for s in infos]).reshape(-1, 4)
            assert np.array_equal(got, G[f"{key}_segments"]), key
            assert np.array_equal(np.stack([s["all_class_probs"].numpy() for s in infos]), G[f"{key}_all_class_probs"])
            assert np.allclose([s["confidence"] for s in infos], G[f"{key}_confidence"], rtol=1e-7)
    # merged stuff: painted with the first segment's id, confidence 0 (helper.py:234-237)
    assert any((G[f"s{si}_i{i}_pan"] > 0).sum() > (G[f"s{si}_i{i}_vox_conf"] > 0).sum()
               for si in range(len(SEEDS)) for i in range(S.N_INSTANCES))


def test_panoptic_inference_default_output_is_unchanged():
    from pasco_b200 import ensemble as E
    ins = _scenes()[0]["instances"][0]
    a = E.panoptic_inference(ins["vox_probs"], ins["query_probs"], OVERLAP, OBJECT_MASK, S.THING_IDS)
    b = E.panoptic_inference(ins["vox_probs"], ins["query_probs"], OVERLAP, OBJECT_MASK, S.THING_IDS, return_confidence=True)
    assert len(a) == 3 and torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert a[2] == [{k: v for k, v in s.items() if k != "all_class_probs"} for s in b[2]]
    assert all("all_class_probs" not in s for s in a[2])


def test_host_logic_matches_the_reference_cpu():
    evs, log = _run(torch.device("cpu"), TORCH_KERNELS)
    _check_tables(log)
    for i, ev in enumerate(evs):
        _check_stats(ev.stats(), i)
    assert math.isnan(evs[1].stats()["ssc"]["empty_ece"])               # instance 1 never predicts empty


def test_gt_panoptic_quirks():
    from pasco_b200.evaluation import gt_panoptic
    masks = torch.zeros(4, 2, 2, 1, dtype=torch.bool)
    masks[0, 0] = True                                                   # stuff 10: cells (0, *)
    masks[1, :, 0] = True                                                # thing 1 overwrites (0, 0)
    masks[2, 1] = True                                                   # stuff 10 again → id 1, overwrites (1, 0)
    masks[3] = True                                                      # label 0 paints nothing
    gid, seg, opens, area = gt_panoptic(torch.tensor([10, 1, 10, 0]), masks, [1])
    assert gid.view(2, 2).tolist() == [[2, 1], [1, 1]]
    assert seg.tolist() == [1, 2, 1, 0] and opens.tolist() == [True, True, False, False] and area.tolist() == [2, 2, 2, 4]


@pytest.mark.gpu
def test_kernel_tables_and_metrics_match_the_reference_gpu():
    from pasco_b200.evaluation import CUDA_KERNELS
    evs, log = _run(torch.device("cuda"), CUDA_KERNELS)
    _check_tables(log)
    for i, ev in enumerate(evs):
        _check_stats(ev.stats(), i)


@pytest.mark.gpu
def test_evaluation_is_bit_identical_run_to_run_gpu():
    from pasco_b200.evaluation import CUDA_KERNELS
    (e1, l1), (e2, l2) = _run(torch.device("cuda"), CUDA_KERNELS), _run(torch.device("cuda"), CUDA_KERNELS)
    for (n1, a1), (n2, a2) in zip(l1, l2):
        assert n1 == n2 and all(torch.equal(x, y) for x, y in zip(a1, a2)), n1
    for a, b in zip(e1, e2):
        sa, sb = a.stats(), b.stats()
        assert repr(sa) == repr(sb)


@pytest.mark.gpu
def test_out_of_range_segment_id_raises_gpu():
    from pasco_b200._lib import PascoError
    from pasco_b200.evaluation import Evaluator
    sc = _scenes()[0]
    ins = sc["instances"][0]
    dev = torch.device("cuda")
    ev = Evaluator(S.K, S.THING_IDS, compute_uncertainty=False)
    pan = torch.full((ins["lin"].numel(),), 7, dtype=torch.int32, device=dev)
    ml = {k: v.to(dev) for k, v in sc["mask_label"].items()}
    with pytest.raises(PascoError):
        ev.add_scene(ins["prob"].to(dev), pan, ins["lin"].to(dev), None, [], sc["semantic_label"].to(dev), ml)
    ev.reset()                                                           # the flag was cleared: a valid scene passes
    ev.add_scene(ins["prob"].to(dev), torch.zeros_like(pan), ins["lin"].to(dev), None, [], sc["semantic_label"].to(dev), ml)
    assert ev.stats()["ssc"]["iou"] > 0


def _compare_with_reference(got, ref, tol=1e-5):
    for k in ("precision", "recall", "iou", "iou_ssc_mean", "empty_ece", "nonempty_ece", "empty_nll", "nonempty_nll"):
        _close(got["ssc"][k], ref["ssc"][k], tol, k)
    assert np.allclose(got["ssc"]["iou_ssc"], ref["ssc"]["iou_ssc"], rtol=0, atol=tol)
    for name in ("All", "Things", "Stuff"):
        for k in ("pq_dagger", "pq", "sq", "rq", "n"):
            _close(got["pq"][name][k], ref["pq"][name][k], tol, f"{name} {k}")
    assert list(got["pq"]["per_class"]) == [int(c) for c in ref["pq"]["per_class"]]
    for k in ("mask_ece", "ins_ece", "ins_nll", "count"):
        _close(got["uncertainty"][k], ref["uncertainty"][k], tol, k)


needs_ref = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "pasco")),
                               reason="no upstream PaSCo package: build() compiles one into oracle/_ref from a checkout")


@pytest.mark.gpu
@needs_ref
def test_benchmark_scale_metrics_equal_the_reference_code_gpu():
    from pasco_b200.evaluation import Evaluator
    from reference_metrics import ReferenceMetrics
    dev = torch.device("cuda")
    sc = S.make_big_scene(0)
    ref = ReferenceMetrics(REF, len(sc["instances"]))
    evs = [Evaluator(S.K, S.THING_IDS, compute_uncertainty=True) for _ in sc["instances"]]
    label = sc["semantic_label"].to(dev)
    ml = {k: v.to(dev) for k, v in sc["mask_label"].items()}
    n_seg = []
    for i, ins in enumerate(sc["instances"]):
        d = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in ins.items()}
        infos = [dict(s, all_class_probs=s["all_class_probs"].to(dev)) for s in d["segments_info"]]
        evs[i].add_scene(d["prob"], d["pan"], d["lin"], d["vox_conf"], infos, label, ml)
        ref.add_scene(i, d["prob"], d["pan"], d["lin"], d["vox_conf"], [dict(s) for s in infos], label, sc["mask_label"])
        n_seg.append(len(infos))
    assert min(n_seg) >= 80
    for i, ev in enumerate(evs):
        _compare_with_reference(ev.stats(), ref.stats(i))


@pytest.mark.gpu
@needs_ref
def test_evaluate_step_end_to_end_gpu():
    from pasco_b200 import ops
    from pasco_b200.evaluation import Evaluator, evaluate_step
    from pasco_b200.net3d import PascoNet
    from pasco_b200.synthetic import make_scene
    from reference_metrics import ReferenceMetrics
    dev = torch.device("cuda")
    ops.set_precision("fp32")
    torch.manual_seed(0)
    M = 3
    net = PascoNet(n_classes=20, n_infers=M, in_channels=283, f=64, num_queries=100).to(dev).eval()
    sc = make_scene((256, 256, 32), 0.05, M, seed=0)
    big = S.make_big_scene(1, n_instances=0)
    d = lambda t: t.to(dev)  # noqa: E731
    batch = dict(sc, in_feats=[d(t) for t in sc["in_feats"]], in_coords=[d(t) for t in sc["in_coords"]],
                 semantic_label_origin=big["semantic_label"].unsqueeze(0).to(dev),
                 mask_label_origin=[{k: d(v) for k, v in big["mask_label"].items()}])
    evs = [Evaluator(20, compute_uncertainty=True) for _ in range(M + 1)]
    # thresholds low enough that the untrained network's queries form segments
    outs = evaluate_step(net, batch, "test", evs, object_mask_threshold=0.0, overlap_threshold=0.0)
    assert len(outs) == M + 1
    ref = ReferenceMetrics(REF, M + 1)
    from pasco_b200.ensemble import ensemble_sem_compl
    with torch.no_grad():
        out = net(batch["in_feats"], batch["in_coords"], sc["global_min_Cs"], sc["global_max_Cs"], sc["min_Cs"],
                  sc["max_Cs"], test=True)
        sem_d = ensemble_sem_compl([(t.F, t.C[:, 1:]) for t in out["sem_logits_pruneds"]], sc["Ts"])
    for i, (pan, lin, conf, infos) in enumerate(outs):
        ref.add_scene(i, sem_d[i], pan, lin, conf, [dict(s) for s in infos], batch["semantic_label_origin"][0],
                      big["mask_label"])
        st = evs[i].stats()
        assert all(math.isfinite(float(st["pq"]["All"][k])) for k in ("pq", "sq", "rq"))
        assert math.isfinite(st["ssc"]["iou"]) and math.isfinite(st["uncertainty"]["ins_nll"])
        _compare_with_reference(st, ref.stats(i))
