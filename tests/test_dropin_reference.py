"""The real drop-in: the UNMODIFIED reference model (`pasco.models.net_panoptic_sparse.Net`, compiled by build() from an
upstream PaSCo checkout into oracle/_ref/, which is not committed) runs on the B200 with `import MinkowskiEngine` /
`torch_scatter` resolving to compat/ → pasco_b200.me → libpasco_sm100.so, and its outputs are compared (a) with the
golden vectors the same reference produced on the CPU oracle and (b) with the engine-native PascoNet on the same
weights and scene.

Reference path exercised: net_panoptic_sparse.py:210-312 → unet3d_sparse_v2.py:216-256 (encoder_v2, dense bottleneck
through nn.Conv3d, decoder_v3 incl. predict_completion_sem_logit / predict_panop, transformer_predictor_v2).
PASCO_REFERENCE (the root of an upstream checkout) overrides oracle/_ref; the tests skip when neither holds `pasco/`.
"""
import json
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("PASCO_REFERENCE") or os.path.join(ROOT, "oracle", "_ref")
sys.path.insert(0, os.path.join(HERE, "golden"))
from recipe import fill_state_dict  # noqa: E402
from test_golden_net import _compare  # noqa: E402

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "pasco")),
                                 reason="no upstream PaSCo package: build() compiles one into oracle/_ref from a checkout")]


def _reference_net(n_infers=1, heavy=False, n_classes=20, in_channels=283):
    for p in (REF, os.path.join(ROOT, "compat")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import MinkowskiEngine as ME
    assert "pasco_b200" in ME.__name__ or "compat" in (ME.__file__ or ""), f"MinkowskiEngine resolved to {ME.__file__}"
    assert ME.SparseTensor.__module__.startswith("pasco_b200.me"), ME.SparseTensor.__module__
    from pasco.models.net_panoptic_sparse import Net
    assert os.path.realpath(sys.modules["pasco.models.net_panoptic_sparse"].__file__).startswith(os.path.realpath(REF))
    freqs = {f"1_{s}": np.ones(n_classes) for s in (1, 2, 4)}
    torch.manual_seed(0)
    net = Net(n_classes=n_classes, class_names=[str(i) for i in range(n_classes)], class_weights=torch.ones(n_classes),
              encoder_dropouts=[0.0] * 3, decoder_dropouts=[0.0] * 3, dense3d_dropout=0.0, n_infers=n_infers,
              class_frequencies=freqs, in_channels=in_channels, num_queries=100, f=64, heavy_decoder=heavy)
    return ME, net


def _forward_reference(ME, net, b, dev, test=False):
    """What Net.step does up to the losses (net_panoptic_sparse.py:314-352), on device tensors."""
    d = lambda t: t.to(dev)  # noqa: E731
    in_coords, in_feats = net.feat([d(t) for t in b["in_feats"]], [d(t) for t in b["in_coords"]])
    x = net.augmenter.merge(ME.SparseTensor(in_feats, in_coords.int()))
    return net(x, 1, {k: d(v) for k, v in b["sem_labels"].items()}, global_min_coords=d(b["global_min_Cs"]),
               global_max_coords=d(b["global_max_Cs"]), min_Cs=[d(t) for t in b["min_Cs"]], max_Cs=[d(t) for t in b["max_Cs"]],
               Ts=[d(t) for t in b["Ts"]], is_predict_panop=True, return_ensemble=False, test=test)


def _rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / b.abs().max())


def test_unmodified_reference_net_on_the_engine_matches_golden_and_pasconet():
    from pasco_b200 import ops
    from pasco_b200.net3d import PascoNet
    from pasco_b200.synthetic import make_scene
    ops.set_precision("fp32")
    man = json.load(open(os.path.join(HERE, "golden", "net_cfg1_manifest.json")))
    gold = np.load(os.path.join(HERE, "golden", "net_cfg1.npz"))
    dev = torch.device("cuda")
    ME, net = _reference_net()
    sd = fill_state_dict(net.state_dict())
    net.load_state_dict(sd)
    net.to(dev).train()
    b = make_scene(man["grid"], man["occ"], 1, seed=man["seed"])
    calls0 = ops.CALLS
    with torch.no_grad():
        out = _forward_reference(ME, net, b, dev)
    assert ops.CALLS - calls0 > 100, "the reference forward did not run on the engine's C-ABI"
    step, report = man["row_step"], {}
    for s in (4, 2, 1):
        lg = out["sem_logits_at_scales"][s][0]
        report[f"sem{s}"] = _compare(f"sem{s}", lg.C, lg.F, gold[f"sem{s}_C"], gold[f"sem{s}_F"], step)
    p = out["panop_predictions"][0]
    report["vox"] = _compare("voxel_logits", p["voxel_logits"].C, p["voxel_logits"].F, gold["vox_C"], gold["vox_F"], step)
    report["query"] = _rel(p["query_logits"][0], gold["query_logits"])
    assert report["query"] <= 1e-3, report
    for i, aux in enumerate(p["aux_outputs"]):
        e = _rel(aux["query_logits"][0], gold[f"aux{i}_query_logits"])
        assert e <= 1e-3, (i, e)
    print("drop-in (unmodified reference on pasco_b200.me) vs golden:", report)

    # (b) the engine-native composition on the same weights and scene agrees with the reference-driven one
    torch.manual_seed(0)
    mine = PascoNet(n_classes=20, n_infers=1, in_channels=283, f=64, num_queries=100)
    mine.load_reference_state_dict({k: v for k, v in sd.items()})
    mine.to(dev).train()
    with torch.no_grad():
        o2 = mine([t.to(dev) for t in b["in_feats"]], [t.to(dev) for t in b["in_coords"]], b["global_min_Cs"],
                  b["global_max_Cs"], b["min_Cs"], b["max_Cs"])
    for s in (4, 2, 1):
        a, c = out["sem_logits_at_scales"][s][0], o2["sem_logits_at_scales"][s][0]
        order = torch.argsort(_keys_of(a.C))
        sym, err = _compare(f"native-vs-dropin sem{s}", c.C, c.F, a.C.cpu()[order].numpy(),
                            a.F.detach().cpu()[order][::step].numpy(), step)
        assert err <= 1e-3


def test_reference_with_attention_hooks_matches_golden():
    """pasco_b200.hooks.install(): the unmodified reference's CrossAttentionLayer / compute_attn_mask run on the xattn
    kernels and the sparse mask instead of nn.MultiheadAttention and the dense [100, X, Y, Z] volume — same golden."""
    from pasco_b200 import ops, hooks
    from pasco_b200.synthetic import make_scene
    ops.set_precision("fp32")
    man = json.load(open(os.path.join(HERE, "golden", "net_cfg1_manifest.json")))
    gold = np.load(os.path.join(HERE, "golden", "net_cfg1.npz"))
    dev = torch.device("cuda")
    ME, net = _reference_net()
    net.load_state_dict(fill_state_dict(net.state_dict()))
    net.to(dev).train()
    assert hooks.install()
    try:
        b = make_scene(man["grid"], man["occ"], 1, seed=man["seed"])
        out = _forward_reference(ME, net, b, dev)
        p = out["panop_predictions"][0]
        report = {"vox": _compare("voxel_logits", p["voxel_logits"].C, p["voxel_logits"].F, gold["vox_C"], gold["vox_F"], man["row_step"]),
                  "query": _rel(p["query_logits"][0], gold["query_logits"])}
        assert report["query"] <= 1e-3, report
        for i, aux in enumerate(p["aux_outputs"]):
            assert _rel(aux["query_logits"][0], gold[f"aux{i}_query_logits"]) <= 1e-3
        (p["voxel_logits"].F.square().mean() + p["query_logits"].square().mean()).backward()
        g = net.transformer_predictor.transformer_cross_attention_layers[1].multihead_attn.in_proj_weight.grad
        assert g is not None and torch.isfinite(g).all() and float(g.abs().max()) > 0
        print("drop-in with attention hooks vs golden:", report)
    finally:
        hooks.uninstall()


def _keys_of(C):
    c = C.long().cpu()
    return ((c[:, 0] + 32768) << 48) | ((c[:, 1] + 32768) << 32) | ((c[:, 2] + 32768) << 16) | (c[:, 3] + 32768)


def test_unmodified_reference_training_step_backward_runs_on_the_engine():
    """fwd + bwd of the unmodified reference network (loss = Σ logits²) — every parameter on the path gets a finite
    gradient through the engine's autograd Functions."""
    from pasco_b200 import ops
    from pasco_b200.synthetic import make_scene
    ops.set_precision("fp32")
    dev = torch.device("cuda")
    ME, net = _reference_net()
    net.load_state_dict(fill_state_dict(net.state_dict()))
    net.to(dev).train()
    b = make_scene((64, 64, 8), 0.05, 1, seed=0)
    out = _forward_reference(ME, net, b, dev)
    loss = sum(lg.F.square().mean() for s in (4, 2, 1) for lg in out["sem_logits_at_scales"][s])
    p = out["panop_predictions"][0]
    loss = loss + p["voxel_logits"].F.square().mean() + p["query_logits"].square().mean()
    loss.backward()
    torch.cuda.synchronize()
    named = [(n, q) for n, q in net.named_parameters() if q.grad is not None]
    assert len(named) > 300, len(named)
    bad = [n for n, q in named if not torch.isfinite(q.grad).all()]
    assert not bad, bad[:5]
    for must in ("unet3d.encoder.s1s2.0.net.0.kernel", "unet3d.dense3d.0.a_conv4.0.weight",
                 "unet3d.decoder_generative.voxel_feats.scale1_infer0.0.kernel", "transformer_predictor.input_projs.2.weight"):
        g = dict(named).get(must)
        assert g is not None and float(g.grad.abs().max()) > 0, must
