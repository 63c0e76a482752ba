"""Seeded synthetic evaluation scenes for tests/test_evaluation.py and make_golden_metrics.py (plain torch, no
reference code).  Each scene has a GT (labels with unknown cells, instance masks) and M + 1 = 4 eval instances, each a
dense class-probability volume plus sparse mask / query probabilities for panoptic inference.  The scenes contain the
cases the metrics treat specially: unknown cells, overlapping GT masks, merged stuff, a GT segment wholly in unknown
cells, a prediction of the wrong class with IoU > 0.5, an unmatched prediction, confidences exactly on bin boundaries and
at 1.0, and an instance whose known cells are never predicted empty (an empty ECE split)."""
import hashlib

import torch

GRID = (64, 64, 16)
K = 20
Q = 12
N_INSTANCES = 4
THING_IDS = [1, 2, 3, 4, 5, 6, 7, 8]


def _box(lo, hi):
    m = torch.zeros(GRID, dtype=torch.bool)
    m[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]] = True
    return m


def make_scene(seed: int):
    g = torch.Generator().manual_seed(seed)
    X, Y, Z = GRID
    cells = X * Y * Z
    # GT masks: (class, box); overlaps, two stuff masks of class 10 (merged), a label-0 mask, one mask in unknown cells
    j = int(torch.randint(0, 4, (1,), generator=g))
    spec = [(0, (0, 0, 0), (64, 64, 2)),
            (1, (10 + j, 10, 2), (22 + j, 20, 8)),
            (2, (30, 8 + j, 2), (40, 22 + j, 10)),
            (10, (0, 40, 0), (32, 64, 4)),
            (3, (44, 30, 3), (56, 40, 9)),
            (10, (32, 40, 0), (64, 64, 4)),
            (12, (20, 30, 5), (36, 44, 12)),
            (5, (14, 14, 4), (20, 24, 8)),              # overlaps the class-1 box and overwrites part of it
            (4, (58, 0, 10), (64, 6, 16)),              # lies wholly in unknown cells
            (9, (40, 50, 6), (60, 62, 14))]
    labels = torch.tensor([s[0] for s in spec], dtype=torch.long)
    masks = torch.stack([_box(lo, hi) for _, lo, hi in spec])
    sem = torch.zeros(cells, dtype=torch.long)
    for i, (c, _, _) in enumerate(spec):
        if c != 0:
            sem[masks[i].view(-1)] = c
    sem = torch.where(torch.rand(cells, generator=g) < 0.03, torch.randint(1, K, (cells,), generator=g), sem)
    label = sem.clone()
    unknown = torch.rand(cells, generator=g) < 0.08
    unknown |= _box((56, 0, 8), (64, 8, 16)).view(-1)
    label[unknown] = 255
    label = label.to(torch.uint8)

    bounds = torch.linspace(0, 1, 16)
    instances = []
    for m in range(N_INSTANCES):
        # dense probabilities: peaked on the (noisy) semantic class, some cells exactly on bin boundaries or one-hot
        tgt = torch.where(torch.rand(cells, generator=g) < 0.8, sem, torch.randint(0, K, (cells,), generator=g))
        if m == 1:
            tgt = torch.where(tgt == 0, torch.randint(1, K, (cells,), generator=g), tgt)   # no empty prediction
        logits = torch.randn(K, cells, generator=g)
        logits[tgt, torch.arange(cells)] += 2.5 + 2 * torch.rand(cells, generator=g)
        prob = torch.softmax(logits, 0)
        pick = torch.randperm(cells, generator=g)[:3000]
        b = bounds[2 + torch.randint(0, 14, (pick.numel(),), generator=g)]               # 2/15 .. 1.0
        col = torch.full((K, pick.numel()), 0.0)
        col += ((1 - b) / (K - 1)).view(1, -1)
        col[tgt[pick], torch.arange(pick.numel())] = b
        prob[:, pick] = col
        onehot = torch.randperm(cells, generator=g)[:2000]
        prob[:, onehot] = 0.0
        prob[tgt[onehot], onehot] = 1.0
        if m == 1:
            prob[0] = 0.0
        # sparse panoptic prediction: rows = cells predicted non-empty; one query per box + a wrong-class copy of the
        # class-3 box, an unmatched box, a second stuff query of class 10
        occ = tgt != 0
        lin = torch.nonzero(occ, as_tuple=True)[0]
        qspec = [(1, 1), (2, 2), (3, 10), (4, 7), (5, 10), (6, 12), (7, 5), (9, 9)]      # (GT mask, predicted class)
        vp = torch.rand(lin.numel(), Q, generator=g) * 0.2
        qp = torch.full((Q, K + 1), 0.01)
        qp[:, K] = 0.5
        for q, (mi, cls) in enumerate(qspec):
            inside = masks[mi].view(-1)[lin]
            vp[inside, q] = 0.6 + 0.4 * torch.rand(int(inside.sum()), generator=g)
            qp[q, cls] = 0.75 + 0.2 * torch.rand(1, generator=g).item()
            qp[q, K] = 0.01
        far = _box((0, 0, 8), (8, 8, 16)).view(-1)[lin]                                      # matches no GT segment
        vp[far, 9] = 0.9
        qp[9, 6] = 0.85
        qp[9, K] = 0.01
        qp = qp / qp.sum(1, keepdim=True)
        instances.append({"prob": prob.view(K, *GRID), "vox_probs": vp, "lin": lin, "query_probs": qp})
    return {"semantic_label": label.view(GRID), "mask_label": {"labels": labels, "masks": masks},
            "instances": instances}


def checksum(scenes) -> str:
    h = hashlib.sha256()
    for s in scenes:
        h.update(s["semantic_label"].numpy().tobytes())
        h.update(s["mask_label"]["masks"].numpy().tobytes())
        for ins in s["instances"]:
            for k in ("prob", "vox_probs", "lin", "query_probs"):
                h.update(ins[k].numpy().tobytes())
    return h.hexdigest()


def calibration_bins(preds: torch.Tensor, target: torch.Tensor, n_bins: int = 15):
    """The binning of torchmetrics' binary_calibration_error (torchmetrics.functional.classification.calibration_error:
    _binning_bucketize with bin_boundaries = torch.linspace(0, 1, n_bins + 1) in the dtype of the confidences;
    confidences = preds, accuracies = target, no folding of p < 0.5).  Restated from its documented source; torchmetrics
    is not a dependency of this project and the restatement has not been run against it.  Returns (count, Σ confidence, Σ accuracy) over n_bins + 1 slots, in float64."""
    conf = preds.float().reshape(-1)
    acc = target.reshape(-1).double()
    bounds = torch.linspace(0, 1, n_bins + 1, dtype=conf.dtype, device=conf.device)
    idx = torch.bucketize(conf, bounds, right=True) - 1
    nb = n_bins + 1
    z = torch.zeros(nb, dtype=torch.float64, device=conf.device)
    count = z.clone().index_add_(0, idx, torch.ones_like(acc))
    sconf = z.clone().index_add_(0, idx, conf.double())
    sacc = z.clone().index_add_(0, idx, acc)
    return count, sconf, sacc


def binary_calibration_error(preds, target, n_bins=15, norm="l1", **_):
    """torchmetrics' binary_calibration_error (l1 norm) from calibration_bins: Σ |acc̄ - conf̄| · count / Σ count, NaN
    for an empty input."""
    assert norm == "l1"
    count, sconf, sacc = calibration_bins(preds, target, n_bins)
    acc_bin = torch.nan_to_num(sacc / count)
    conf_bin = torch.nan_to_num(sconf / count)
    return torch.sum(torch.abs(acc_bin - conf_bin) * (count / count.sum())).float()


def make_big_scene(seed: int = 0, grid=(256, 256, 32), n_segments: int = 100, n_instances: int = 4):
    """A benchmark-scale scene (default 256 x 256 x 32, K = 20) with `n_segments` GT box masks and, per eval instance,
    a dense probability volume and a panoptic prediction given directly as rows (pan, lin, vox_conf, segments_info):
    each GT box is predicted as a jittered box, some with the wrong class."""
    g = torch.Generator().manual_seed(seed)
    X, Y, Z = grid
    cells = X * Y * Z
    labels = torch.randint(1, K, (n_segments,), generator=g)
    lo = torch.stack([torch.randint(0, X - 16, (n_segments,), generator=g), torch.randint(0, Y - 16, (n_segments,), generator=g),
                      torch.randint(0, Z - 6, (n_segments,), generator=g)], 1)
    ext = torch.stack([torch.randint(4, 16, (n_segments,), generator=g), torch.randint(4, 16, (n_segments,), generator=g),
                       torch.randint(2, 6, (n_segments,), generator=g)], 1)
    masks = torch.zeros(n_segments, X, Y, Z, dtype=torch.bool)
    sem = torch.zeros(X, Y, Z, dtype=torch.long)
    for i in range(n_segments):
        (a, b, c), (u, v, w) = lo[i].tolist(), (lo[i] + ext[i]).tolist()
        masks[i, a:u, b:v, c:w] = True
        sem[a:u, b:v, c:w] = labels[i]
    label = sem.view(-1).clone()
    label[torch.rand(cells, generator=g) < 0.15] = 255
    bounds = torch.linspace(0, 1, 16)
    instances = []
    for _ in range(n_instances):
        tgt = torch.where(torch.rand(cells, generator=g) < 0.85, sem.view(-1), torch.randint(0, K, (cells,), generator=g))
        logits = torch.randn(K, cells, generator=g)
        logits[tgt, torch.arange(cells)] += 3.0
        prob = torch.softmax(logits, 0)
        pick = torch.randperm(cells, generator=g)[:20000]
        prob[:, pick] = 0.0
        prob[tgt[pick], pick] = bounds[2 + torch.randint(0, 14, (pick.numel(),), generator=g)]
        pan = torch.zeros(X, Y, Z, dtype=torch.int32)
        conf = torch.zeros(X, Y, Z)
        infos = []
        for i in range(n_segments):
            d = torch.randint(-2, 3, (3,), generator=g)
            a, b, c = (lo[i] + d).clamp(min=0).tolist()
            u, v, w = (lo[i] + ext[i] + d).tolist()
            pan[a:u, b:v, c:w] = i + 1
            conf[a:u, b:v, c:w] = 0.3 + 0.7 * torch.rand(pan[a:u, b:v, c:w].shape, generator=g)
            cls = int(labels[i]) if torch.rand(1, generator=g).item() < 0.8 else int(torch.randint(1, K, (1,), generator=g))
            acp = torch.softmax(torch.randn(K + 1, generator=g), 0)
            infos.append({"id": i + 1, "isthing": cls in THING_IDS, "category_id": cls, "query_id": i,
                          "confidence": float(acp.max()), "all_class_probs": acp})
        # the last segments' boxes may cover whole earlier ones: keep the ids that are still painted
        lin = torch.nonzero(pan.view(-1) != 0, as_tuple=True)[0]
        present = set(torch.unique(pan).tolist())
        infos = [s for s in infos if s["id"] in present]
        instances.append({"prob": prob.view(K, *grid), "pan": pan.view(-1)[lin], "lin": lin, "vox_conf": conf.view(-1)[lin],
                          "segments_info": infos})
    return {"semantic_label": label.view(grid).to(torch.uint8), "mask_label": {"labels": labels, "masks": masks},
            "instances": instances}
