"""Evaluation cost per scene: the engine's device evaluator against the reference's own metric code on the same outputs.

    python tools/eval_bench.py --out DIR [--reps 20]

One benchmark-scale scene (tests/golden/metrics_scenes.make_big_scene: 256 x 256 x 32, K = 20, ~100 segments) with
M + 1 = 4 eval instances, test mode (uncertainty metrics on).  Times, per scene (all 4 instances):
  - evaluation.Evaluator.add_scene on the device (CUDA events, after warm-up), including its one device→host copy;
  - the reference's SSCMetrics / pq_compute_single_core / find_matched_segment / UncertaintyMetrics through
    Net.evaluate_all (tests/golden/reference_metrics.py, from oracle/_ref), host clock around work ending in a device
    synchronise, its own device→host copies included; reported as missing when oracle/_ref is absent;
  - k_eval_ssc alone (CUDA events over many launches) with the bytes it must read (K x cells x 4 + cells) over that time
    against 7.7 TB/s.  The 168 MB volume is larger than the 126 MB L2, so repeated launches stream it from HBM.
Writes one JSON line to DIR/eval_bench.json and prints it; card name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests", "golden")]
HBM_BYTES_PER_S = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for eval_bench.json")
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "eval_bench measures on the GPU"
    from pasco_b200 import build
    build.build()
    from pasco_b200 import ops
    from pasco_b200.evaluation import Evaluator, calibration_bounds
    import metrics_scenes as S
    dev = torch.device("cuda")
    sc = S.make_big_scene(0)
    label = sc["semantic_label"].to(dev)
    ml = {k: v.to(dev) for k, v in sc["mask_label"].items()}
    ins = []
    for x in sc["instances"]:
        d = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in x.items()}
        d["segments_info"] = [dict(s, all_class_probs=s["all_class_probs"].to(dev)) for s in d["segments_info"]]
        ins.append(d)

    def device_scene(evs):
        for e, d in zip(evs, ins):
            e.add_scene(d["prob"], d["pan"], d["lin"], d["vox_conf"], d["segments_info"], label, ml)

    evs = [Evaluator(S.K, S.THING_IDS, compute_uncertainty=True) for _ in ins]
    for _ in range(3):
        device_scene(evs)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.reps):
        device_scene(evs)
    e1.record()
    torch.cuda.synchronize()
    dev_ms = e0.elapsed_time(e1) / a.reps
    stats = evs[-1].stats()

    # k_eval_ssc alone
    prob, lab = ins[0]["prob"].reshape(S.K, -1), label.reshape(-1)
    bounds = calibration_bounds(15, dev)
    counts = torch.zeros(S.K * S.K + 64, dtype=torch.int64, device=dev)
    sums = torch.zeros(34, dtype=torch.float64, device=dev)
    for _ in range(5):
        ops.eval_ssc(prob, lab, bounds, counts, sums)
    n_launch = 200
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n_launch):
        ops.eval_ssc(prob, lab, bounds, counts, sums)
    e1.record()
    torch.cuda.synchronize()
    ssc_us = e0.elapsed_time(e1) * 1e3 / n_launch
    nbytes = prob.numel() * 4 + lab.numel()

    ref_root = os.environ.get("PASCO_REFERENCE") or os.path.join(ROOT, "oracle", "_ref")
    ref = {"status": "missing: no upstream package under oracle/_ref"}
    if os.path.isdir(os.path.join(ref_root, "pasco")):
        from reference_metrics import ReferenceMetrics
        rm = ReferenceMetrics(ref_root, len(ins))

        def ref_scene():
            for i, d in enumerate(ins):
                rm.add_scene(i, d["prob"], d["pan"], d["lin"], d["vox_conf"], [dict(s) for s in d["segments_info"]],
                             label, sc["mask_label"])
            torch.cuda.synchronize()

        ref_scene()                                                    # warm-up
        times = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ref_scene()
            times.append((time.perf_counter() - t0) * 1e3)
        ref = {"status": "ok", "ms_per_scene": round(min(times), 2), "ms_per_scene_all": [round(t, 2) for t in times]}
    res = {"what": "evaluation per scene (4 eval instances, test mode, uncertainty on)", "grid": [256, 256, 32],
           "K": S.K, "segments_per_instance": [len(d["segments_info"]) for d in ins], "card": card(),
           "device_evaluator_ms_per_scene": round(dev_ms, 3), "reference_metric_code": ref,
           "speedup": round(ref["ms_per_scene"] / dev_ms, 1) if ref["status"] == "ok" else None,
           "k_eval_ssc": {"us": round(ssc_us, 2), "bytes": nbytes, "TB_per_s": round(nbytes / ssc_us / 1e6, 3),
                          "share_of_7.7TB_per_s": round(nbytes / (ssc_us * 1e-6) / HBM_BYTES_PER_S, 3)},
           "ensemble_pq_all": {k: float(v) for k, v in stats["pq"]["All"].items()}}
    os.makedirs(a.out, exist_ok=True)
    line = json.dumps(res)
    with open(os.path.join(a.out, "eval_bench.json"), "w") as f:
        f.write(line + "\n")
    print(line, flush=True)


if __name__ == "__main__":
    main()
