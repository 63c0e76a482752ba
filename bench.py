#!/usr/bin/env python
"""bench.py — scenes/sec (256×256×32 voxels @10 % occupancy) forward+backward, the BASELINE.json metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision fp32|bf16] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one synthetic scene per GPU: point voxeliser → Net3D sparse
U-Net → mask transformer (M=1, f=64, 100 queries, train-mode BatchNorm, decoder caps active) → losses →
backward (N>1: gradient buckets all-reduced over NCCL while it runs) → fused AdamW step.  Weak scaling: one scene
per GPU per step, `value` = N·K scenes ÷ max-over-ranks device time.

Two timed regions, both bracketed by barrier + cuda.synchronize and CUDA events:
  value : inputs already resident in HBM (fresh scene every step, so coordinate maps are rebuilt);
  e2e   : same K steps through the same public call with the step's inputs coming from pinned host
          memory (H2D inside the region, issued one step ahead on a copy stream) and the loss read back
          (asynchronous D2H into pinned memory) every step.
`--impl reference` times the CPU restatement of the MinkowskiEngine algorithm (oracle/) on the host
cores on a bounded crop of the same workload (ME 0.5.4 itself is not installable offline, BASELINE.md §2).
`--dump-outputs DIR` writes what the last timed step computed as DIR/<name>.npy (see dump_outputs); scenes and initial
weights are seeded, so runs with the same arguments get the same inputs and two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")   # scene sizes vary step to step
import faulthandler  # noqa: E402

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

faulthandler.enable()
_T0 = time.time()


def log(msg):
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench {time.time() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)

GRID, OCC, IN_CH, N_CLASSES = (256, 256, 32), 0.10, 283, 20
SETTLE = 8          # extra untimed steps right before the first timed region (on top of --warmup): twice through the scene pool
METRIC = "scenes/sec (256x256x32 voxels @10% occ) fwd+bwd"
# --shape: the two dataset shapes of BASELINE.json's configs (SemanticKITTI: net_panoptic_sparse.py:51; KITTI-360:
# train_kitti360.py:115,152 — 19 classes, 8-wide point features, 8 % occupancy in configs[4])
SHAPES = {"semkitti": dict(occ=0.10, in_ch=283, n_classes=20), "kitti360": dict(occ=0.08, in_ch=8, n_classes=19)}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0)), "measured"
    return 6650.0, 1400.0, "fallback"


NCU_FILE = "r02_ncu_conv_planes.json"


def _kernel_name(kind, meta):
    path = meta.get("path", "regs")
    if path == "planes":
        return "k_wgrad_pl" if kind == "wgrad" else "k_conv_pl"
    if path == "simt":
        return "k_wgrad_simt" if kind == "wgrad" else "k_conv_simt"
    return "k_wgrad_tc" if kind == "wgrad" else "k_conv_tc"


def _ncu_traffic(kind, meta):
    """dram__bytes_read.sum + dram__bytes_write.sum (bytes) per launch of the dominant kernel from the committed
    ncu --set full capture of the same layer shape (profiles/r02_ncu_conv_planes.json: N=1.05 M rows, C=64, bf16x3);
    None if the dominant group is another shape or the capture is absent."""
    if not (meta["Cin"] == 64 and meta["Cout"] == 64 and meta["K"] == 27 and 0.9e6 < meta["n_out"] < 1.2e6 and meta["precision"] == 3):
        return None
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", NCU_FILE)))
        want = _kernel_name(kind, meta)
        for k in d["kernels"]:
            if want in k["kernel"]:
                return float(k["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop_evt.is_set():
            try:
                r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                   capture_output=True, text=True, timeout=5)
                self.rows.append([x.strip() for x in r.stdout.strip().split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def to_device(scene, dev, non_blocking=True):
    out = {}
    for k, v in scene.items():
        if isinstance(v, torch.Tensor):
            out[k] = v.to(dev, non_blocking=non_blocking)
        elif isinstance(v, list) and v and isinstance(v[0], torch.Tensor):
            out[k] = [t.to(dev, non_blocking=non_blocking) for t in v]
        elif isinstance(v, dict):
            out[k] = {a: b.to(dev, non_blocking=non_blocking) for a, b in v.items()}
        else:
            out[k] = v
    return out


def _tensors(scene):
    for v in scene.values():
        if isinstance(v, torch.Tensor):
            yield v
        elif isinstance(v, list):
            yield from (t for t in v if isinstance(t, torch.Tensor))
        elif isinstance(v, dict):
            yield from (t for t in v.values() if isinstance(t, torch.Tensor))


def pin(scene):
    out = {}
    for k, v in scene.items():
        if isinstance(v, torch.Tensor):
            out[k] = v.pin_memory()
        elif isinstance(v, list) and v and isinstance(v[0], torch.Tensor):
            out[k] = [t.pin_memory() for t in v]
        elif isinstance(v, dict):
            out[k] = {a: b.pin_memory() for a, b in v.items()}
        else:
            out[k] = v
    return out


def h2d_bytes(scene):
    n = 0
    for k in ("in_feats", "in_coords"):
        n += sum(t.numel() * t.element_size() for t in scene[k])
    n += sum(t.numel() * t.element_size() for t in scene["sem_labels"].values())
    n += scene["mask_classes"].numel() * 8
    return n


DUMP_BUDGET = 64 << 20          # bytes written by --dump-outputs, all files together
DUMP_PARAM_SAMPLE = 1 << 20     # entries of the flattened parameters (and of their gradients) written


def _named_outputs(prefix, v, acc):
    """Flattens the network's output structure into {"sem_logits_at_scales.4.0": tensor-or-SparseTensor, ...}."""
    if isinstance(v, dict):
        for k, x in v.items():
            _named_outputs(f"{prefix}{k}.", x, acc)
    elif isinstance(v, (list, tuple)):
        for i, x in enumerate(v):
            _named_outputs(f"{prefix}{i}.", x, acc)
    elif isinstance(v, torch.Tensor) or (hasattr(v, "F") and hasattr(v, "C")):
        acc[prefix[:-1]] = v


def dump_outputs(path, out, loss, params):
    """Writes one step's results as path/<name>.npy: `loss` (float64), every dense output tensor (float32), and for every
    sparse output `<name>.coords` (float64 [R, 4], batch x y z) and `<name>.feats` (float32 [R, C]).  Sparse rows are sorted
    by coordinate; a large output keeps the rows whose coordinates hash lowest, so two builds keep the same voxels where
    their coordinate sets agree.  `params_sample` / `grads_sample` (float32) are the parameters after the optimiser step
    and their gradients at 2^20 positions of the flattened parameter list drawn with a fixed seed.

    The dumped step follows W + SETTLE + 2K optimiser steps, and AdamW and the argmax pruning amplify any difference in
    the last bit.  The engine's float reductions sum their partials in a fixed order; the BatchNorm statistics still
    accumulate in float64 atomics, whose order can change the float64 sum's last bit but only rarely the float result.
    Two runs with the same arguments on the same GPU therefore normally write the same arrays."""
    named = {}
    _named_outputs("", out, named)
    sparse = {k: v for k, v in named.items() if not isinstance(v, torch.Tensor)}
    dense = {k: v for k, v in named.items() if isinstance(v, torch.Tensor)}
    # rows per sparse output such that they fit the budget left by the loss, the dense outputs and the two samples
    fixed = 8 + sum(4 * v.numel() for v in dense.values()) + 2 * 4 * DUMP_PARAM_SAMPLE
    row_bytes = sum(8 * 4 + 4 * v.F.shape[1] for v in sparse.values())
    max_rows = max(1, (DUMP_BUDGET - fixed) // max(row_bytes, 1))
    arrays = {"loss": loss.detach().double().cpu().numpy().reshape(1)}
    for k, v in dense.items():
        arrays[k] = v.detach().float().cpu().numpy()
    for k, v in sparse.items():
        c = v.C.detach().long().cpu()
        key = (((c[:, 0] + 32768) << 48) | ((c[:, 1] + 32768) << 32) | ((c[:, 2] + 32768) << 16) | (c[:, 3] + 32768)).numpy()
        rows = np.arange(len(key))
        if len(key) > max_rows:
            h = key.astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)       # wraps mod 2^64: a fixed scramble of the key
            rows = np.argpartition(h, max_rows - 1)[:max_rows]
        rows = rows[np.argsort(key[rows], kind="stable")]
        arrays[f"{k}.coords"] = c.numpy()[rows].astype(np.float64)
        arrays[f"{k}.feats"] = v.F.detach().float().cpu().numpy()[rows]
    flat_p = torch.cat([p.detach().reshape(-1).float() for p in params])
    flat_g = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).detach().reshape(-1).float() for p in params])
    idx = torch.randint(0, flat_p.numel(), (DUMP_PARAM_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort()[0]
    arrays["params_sample"] = flat_p[idx.to(flat_p.device)].cpu().numpy()
    arrays["grads_sample"] = flat_g[idx.to(flat_g.device)].cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_BUDGET, f"--dump-outputs: {total} bytes > {DUMP_BUDGET}"
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, f"{k}.npy"), a)
    return total, len(arrays)


# ------------------------------------------------------------------------------------------------------------
def run_ours(a):
    from pasco_b200 import build
    build.build()
    from pasco_b200 import ops
    from pasco_b200.net3d import PascoNet
    from pasco_b200.losses import total_loss
    from pasco_b200.synthetic import make_scene
    from pasco_b200 import parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — pasco_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ops.set_precision(a.precision)
    shp = SHAPES[a.shape]
    OCC, IN_CH, N_CLASSES = shp["occ"], shp["in_ch"], shp["n_classes"]
    M, ACC = a.m, max(1, a.accum)

    torch.manual_seed(0)
    net = PascoNet(n_classes=N_CLASSES, n_infers=M, in_channels=IN_CH, f=64, num_queries=100,
                   heavy_decoder=a.heavy_decoder).to(dev).train()
    if world > 1:
        n_sync = parallel.enable_sync_batchnorm(net)     # Trainer(sync_batchnorm=True), scripts/train.py:216
        log(f"SyncBatchNorm on {n_sync} fused BN layers")
    params = [p for p in net.parameters() if p.requires_grad]
    opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=1e-4, fused=True)
    # every scene of the pool is seen by a warm-up step, so that the caching allocator holds blocks of every size before
    # the timed regions (a first-touch cudaMalloc synchronises the device)
    n_pool = max(1, min(a.pool, a.warmup * ACC))
    host_scenes = [pin(make_scene(GRID, OCC, M, IN_CH, N_CLASSES, seed=sd, clustered=a.occupancy == "clustered"))
                   for sd in parallel.scene_seeds(rank, world, n_pool)]
    dev_scenes = [to_device(s, dev) for s in host_scenes]
    torch.cuda.synchronize()
    # the reference's DDP gradient averaging (scripts/train.py:213): 64 MB buckets all-reduced while backward continues
    reducer = parallel.GradReducer(params, bucket_mb=a.bucket_mb) if world > 1 else None
    kept = {}                   # outputs of the last timed step, for --dump-outputs

    def step(scene, micro=0, keep=False):
        """One micro-step (one MIMO group of M scenes); the optimiser step closes on the last of ACC micro-steps
        (gradient accumulation, scripts/train.py:62,203: `--accum_batch`)."""
        out = net(scene["in_feats"], scene["in_coords"], scene["global_min_Cs"], scene["global_max_Cs"],
                  scene["min_Cs"], scene["max_Cs"])
        loss = total_loss(out, scene, N_CLASSES, net.class_frequencies)
        if ACC > 1:
            loss = loss / ACC
        if keep:
            kept.update(out=out, loss=loss)
        last = micro == ACC - 1
        if micro == 0:
            if reducer is not None:
                reducer.zero_grad()
            else:
                opt.zero_grad(set_to_none=True)
        if reducer is not None and ACC > 1:
            reducer.rearm(sync=last)
        loss.backward()
        if last:
            if reducer is not None:
                reducer.finish()
            torch.nn.utils.clip_grad_norm_(params, 0.5)
            opt.step()
        return loss

    copy_stream = torch.cuda.Stream(device=dev)
    loss_host = torch.zeros(max(a.steps, 1), dtype=torch.float32).pin_memory()

    def timed(n_steps, from_host, keep_last=False):
        gc.collect()
        gc.disable()            # no collector pauses inside the timed region (collected between regions)
        try:
            return _timed(n_steps, from_host, keep_last)
        finally:
            gc.enable()

    def _timed(n_steps, from_host, keep_last):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = None
        if from_host:
            # the input pipeline a training loop would run: step i+1's scene is copied from pinned host memory on a
            # side stream while step i computes, and every step's loss is read back asynchronously into pinned
            # memory (all copies are issued, and complete, inside the timed region)
            main = torch.cuda.current_stream()

            def prefetch(i):
                with torch.cuda.stream(copy_stream):
                    sc = to_device(host_scenes[i % n_pool], dev)
                    for t in _tensors(sc):
                        t.record_stream(main)
                    ev = torch.cuda.Event()
                    ev.record(copy_stream)
                return sc, ev

            nxt = prefetch(0)
            for i in range(n_steps * ACC):
                sc, ev = nxt
                main.wait_event(ev)
                if i + 1 < n_steps * ACC:
                    nxt = prefetch(i + 1)
                ls = step(sc, i % ACC, keep=keep_last and i == n_steps * ACC - 1).detach()
                if i % ACC == ACC - 1:
                    loss_host[(i // ACC) % loss_host.shape[0]].copy_(ls, non_blocking=True)   # D2H read of the result
        else:
            for i in range(n_steps * ACC):
                last = step(dev_scenes[i % n_pool], i % ACC)
        e1.record()
        torch.cuda.synchronize()
        if from_host:
            last = float(loss_host[(n_steps - 1) % loss_host.shape[0]])
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), last

    # map the allocator's address range once, outside the timed regions: the per-step working set (~20 GB, sizes differ
    # from scene to scene) otherwise grows by cuMemMap calls whenever a step needs a block that is not cached yet
    reserve = torch.empty(int(os.environ.get("PASCO_BENCH_RESERVE_GB", "40")) << 30, dtype=torch.uint8, device=dev)
    del reserve
    torch.cuda.reset_peak_memory_stats(dev)
    gc.collect()
    gc.freeze()
    log(f"model + {n_pool} scenes ready")
    for i in range(a.warmup * ACC):
        faulthandler.dump_traceback_later(240, exit=False)
        step(dev_scenes[i % n_pool], i % ACC)
        torch.cuda.synchronize()
        faulthandler.cancel_dump_traceback_later()
        log(f"warm-up step {i} done, peak mem {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB")
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    # two more untimed steps right before each timed region ("settle"): the first steps after the allocator reservation /
    # after NCCL's first bucketed all-reduces still pay one-time costs (cuMemMap of new block sizes, channel set-up) that
    # showed up as a 20 % slower first region at N = 2
    for i in range(SETTLE * ACC):
        step(dev_scenes[i % n_pool], i % ACC)
    calls0 = ops.CALLS
    ms, _ = timed(a.steps, from_host=False)
    launches = ops.CALLS - calls0
    log(f"device-resident region: {ms / a.steps:.1f} ms/step")
    # untimed: one pass of the input pipeline so that the copy stream's allocator pool holds blocks of every scene size
    # (a first-touch cudaMalloc inside the timed region would synchronise the device)
    main_stream = torch.cuda.current_stream()
    with torch.cuda.stream(copy_stream):
        warm = [to_device(host_scenes[i % n_pool], dev) for i in range(min(n_pool, a.steps))]
        for sc in warm:
            for t in _tensors(sc):
                t.record_stream(main_stream)
    torch.cuda.synchronize()
    del warm
    ms_e2e, _ = timed(a.steps, from_host=True, keep_last=a.dump_outputs is not None)
    log(f"e2e region: {ms_e2e / a.steps:.1f} ms/step")
    if a.dump_outputs is not None and rank == 0:
        # before the profiled step below, which would replace the gradients and update the parameters again
        n_bytes, n_files = dump_outputs(a.dump_outputs, kept["out"], kept["loss"], params)
        log(f"wrote {n_files} arrays ({n_bytes / 2**20:.1f} MiB) of the last timed step to {a.dump_outputs}")
    kept.clear()
    clocks = sampler.stop() if sampler else None
    # per-launch CUDA events of the conv kernels (the roofline block) come from ONE extra step of the same workload run
    # right after the timed regions (same clocks, same allocator state): recording ~260 event pairs and the pair counts
    # inside a timed region cost 5-20 ms/step of host time in round 1 and made `value` slower than `e2e`
    ops.PROFILE = []
    for j in range(ACC):
        step(dev_scenes[(a.steps * ACC + j) % n_pool], j)
    torch.cuda.synchronize()
    prof, ops.PROFILE = ops.PROFILE, None
    prof_steps = 1
    ops.PAIR_COUNTS.clear()

    # ---- roofline of the dominant kernel (per-launch CUDA-event durations recorded inside the timed region) ----
    groups = {}
    for kind, e_a, e_b, m in prof:
        key = (kind, m["n_out"] // 50000, m["K"], m["Cin"], m["Cout"], m.get("path"))
        g = groups.setdefault(key, {"ms": 0.0, "n": 0, "flops": 0.0, "bytes": 0.0, "kind": kind, "meta": m})
        pairs = float(m["pairs"].item()) if m.get("pairs") is not None else float(m["n_out"]) * (m["K"] if m["K"] > 1 else 1)
        g["ms"] += e_a.elapsed_time(e_b)
        g["n"] += 1
        g["flops"] += 2.0 * pairs * m["Cin"] * m["Cout"]
        g["bytes"] += 4.0 * (m["n_in"] * m["Cin"] + m["n_out"] * m["Cout"]) + 4.0 * m["K"] * m["Cin"] * m["Cout"] + 8.0 * pairs
    conv_ms = sum(g["ms"] for g in groups.values())
    if rank == 0 and os.environ.get("PASCO_BENCH_GROUPS"):
        for key, g in sorted(groups.items(), key=lambda kv: -kv[1]["ms"])[:40]:
            log(f"  conv group {g['kind']:5s} n_out~{g['meta']['n_out']:8d} K={g['meta']['K']:3d} {g['meta']['Cin']:4d}->{g['meta']['Cout']:4d}: "
                f"{g['n']:3d} launches, {g['ms'] / prof_steps:7.2f} ms/step, {g['flops'] / g['ms'] / 1e9:6.1f} useful TFLOP/s")
    hbm_peak, tf_peak, peak_src = _peaks()
    roof = None
    if groups:
        top = max(groups.values(), key=lambda g: g["ms"])
        per_launch_ms = top["ms"] / top["n"]
        ach_tf = top["flops"] / top["n"] / per_launch_ms / 1e9
        ach_gb = top["bytes"] / top["n"] / per_launch_ms / 1e6
        m = top["meta"]
        roof = {"kernel": f"{_kernel_name(top['kind'], m)}<{m['precision']}> {top['kind']} K={m['K']} {m['Cin']}->{m['Cout']} n_out~{m['n_out']}",
                "bound": "tensor", "achieved": round(ach_tf, 2), "peak": tf_peak, "unit": "TFLOP/s",
                "frac": round(ach_tf / tf_peak, 4), "traffic": _ncu_traffic(top["kind"], m),
                "traffic_source": f"dram__bytes_read.sum + dram__bytes_write.sum per launch, profiles/{NCU_FILE} (same layer shape)",
                "algorithmic_bytes_per_launch": round(top["bytes"] / top["n"]), "peak_source": peak_src,
                "launch_ms": round(per_launch_ms, 4), "launches": top["n"],
                "algorithmic": "flops = 2*pairs*Cin*Cout per launch (useful MACs; bf16x3 issues 3x that on the tensor pipe)",
                "tensor_issued_TFLOPs": round(ach_tf * (3 if m["precision"] == 3 else 1), 2),
                "tensor_issued_frac": round(ach_tf * (3 if m["precision"] == 3 else 1) / tf_peak, 4),
                "hbm_achieved_GBs": round(ach_gb, 1), "hbm_frac": round(ach_gb / hbm_peak, 4),
                "share_of_step": round(top["ms"] / (ms / a.steps * prof_steps), 3),
                "all_conv_share_of_step": round(conv_ms / (ms / a.steps * prof_steps), 3),
                "events": "per-launch CUDA events of one extra step run right after the timed regions (same workload)"}

    if rank == 0:
        scenes_per_step = world * ACC * M          # a MIMO group holds M scenes (one per subnet), ACC groups per optimiser step
        default_mode = a.shape == "semkitti" and M == 1 and ACC == 1 and not a.heavy_decoder and a.occupancy == "uniform"
        workload = ("configs[1] shape: 256x256x32 @10% occ, full PaSCo (Net3D + MaskPLS 100 queries, M=1, f=64), "
                    "fwd+bwd+AdamW, 1 scene/GPU/step, train-mode caps 25k/120k/400k") if default_mode else (
            f"256x256x32 @{OCC:.0%} occ ({a.occupancy}) {a.shape} shape ({N_CLASSES} classes, {IN_CH}-wide point features), full PaSCo M={M}"
            f"{' heavy decoder' if a.heavy_decoder else ''}, f=64, fwd+bwd+AdamW, {ACC} MIMO group(s) of {M} scene(s) per GPU per "
            f"optimiser step (gradient accumulation), global batch {scenes_per_step} scenes")
        line = {"metric": METRIC, "value": round(scenes_per_step * a.steps / (ms / 1e3), 4), "unit": "scenes/s", "n_gpus": world,
                "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(ms / a.steps, 3), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32 (bf16x3 split tensor-core MMA, fp32 accumulate)"
                if a.precision == "fp32" else "bf16 operands, fp32 accumulate", "data": "synthetic",
                "config": {"workload": workload, "global_batch": scenes_per_step, "accum": ACC, "n_infers": M, "shape": a.shape,
                           "loss": "CE+Lovasz completion @3 scales + Hungarian set loss (class CE, focal, dice, 3 aux levels)",
                           "parallelism": f"dp{world}", "l2": "inputs larger than L2: per-step working set (>4 GB of activations) >> 126 MB",
                           "scene_pool": n_pool, "random_init_weights": True, "settle_steps": SETTLE},
                "e2e": {"value": round(scenes_per_step * a.steps / (ms_e2e / 1e3), 4), "unit": "scenes/s",
                        "h2d_bytes_per_step": h2d_bytes(host_scenes[0]) * ACC, "d2h_bytes_per_step": 4,
                        "ms_per_step": round(ms_e2e / a.steps, 3)},
                "gpu_launches": launches, "clocks": clocks, "roofline": roof}
        if world == 1 and not a.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(a.cpu_seconds)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------
def cpu_baseline(_budget_s: float = 20.0):
    """CPU restatement of the ME algorithm (oracle/) on THE fixed crop of the same workload (net_oracle.CROP_GRID, the same
    crop `--impl reference` times), all host cores: 1 warm-up + 3 timed passes, median and spread."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import net_oracle
    cores = min(os.cpu_count(), 32)     # the per-offset gather/GEMM/scatter loop stops scaling beyond ~32 threads
    torch.set_num_threads(cores)
    log(f"cpu baseline on {cores} threads ...")
    r = net_oracle.time_crop(repeats=3, warmup=1)
    return {"value": round(r["scenes_per_s"], 6), "unit": "scenes/s", "cores": cores, "kind": "port",
            "sample": r["sample"], "seconds_per_sample": r["seconds"], "times": r["times"], "spread": r["spread"],
            "note": "CPU restatement of the MinkowskiEngine 0.5.4 algorithm (ME not installable offline)"}


def run_reference(a):
    """The reference arm: the CPU restatement of the reference's MinkowskiEngine path on the host cores.  One STEP = one
    forward+backward(+losses) pass over the fixed 1/16-scene crop (a bounded sample of config.workload); W warm-up
    (at least 1, at most 2) and exactly K timed steps.
    value = (1/16 scene) / median step time — the linear-in-voxels scaling is stated in config.workload;
    `--ref-full-scene` adds ONE unscaled full-scene pass (minutes) as `full_scene`."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import net_oracle
    cores = min(os.cpu_count(), 32)
    torch.set_num_threads(cores)
    n_warm = max(1, min(a.warmup, 2))
    r = net_oracle.time_crop(repeats=a.steps, warmup=n_warm)
    v = r["scenes_per_s"]
    line = {"impl": "reference", "metric": METRIC, "value": round(v, 6), "unit": "scenes/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": n_warm,
            "ms_per_step": round(r["seconds"] * 1e3, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1] shape: 256x256x32 @10% occ, full PaSCo fwd+bwd+losses (M=1, f=64); each STEP is a "
                                   "bounded sample = one 64x64x32 crop (1/16 scene, caps scaled 1/16); value = 1/(16 x median "
                                   "step time), assuming cost linear in voxels",
                       "parallelism": f"cpu x{cores} threads", "scene_fraction_per_step": 1.0 / r["div"]},
            "cpu_baseline": {"value": round(v, 6), "unit": "scenes/s", "cores": cores, "kind": "port",
                             "sample": r["sample"],
                             "times": r["times"], "spread": r["spread"]},
            "e2e": {"value": round(v, 6), "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if a.ref_full_scene:
        f = net_oracle.time_full_scene()
        line["full_scene"] = {"value": round(f["scenes_per_s"], 6), "unit": "scenes/s", "seconds": f["seconds"], "sample": f["sample"]}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--pool", type=int, default=4, help="distinct synthetic scenes cycled through")
    ap.add_argument("--shape", default="semkitti", choices=sorted(SHAPES), help="dataset shape (classes / point-feature width / occupancy)")
    ap.add_argument("--m", type=int, default=1, help="MIMO subnets per network (n_infers); a step then covers M scenes per group")
    ap.add_argument("--accum", type=int, default=1, help="MIMO groups per GPU per optimiser step (gradient accumulation)")
    ap.add_argument("--heavy-decoder", action="store_true")
    ap.add_argument("--occupancy", default="uniform", choices=["uniform", "clustered"],
                    help="uniform = Bernoulli occupancy (BASELINE configs); clustered = ground slab + boxes, same voxel count")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--bucket-mb", type=float, default=64.0, help="gradient all-reduce bucket size (N > 1)")
    ap.add_argument("--ref-full-scene", action="store_true", help="--impl reference: also time one unscaled full scene")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32/float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
