#!/usr/bin/env python
"""bench.py -- person-crops/s of the ViTPose crop path on N x B200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      (the CPU oracle port of the reference path, host cores)
    python bench.py ... --dump-outputs DIR    (also writes the last timed step's keypoints + argmax as DIR/*.npy)

A step = one pass of the hot path over one batch of synthetic crops per GPU:
    crops f32 [B,3,256,192] (resident in HBM) -> ViT-B -> head -> heatmaps -> decode -> keypoints [B,K,3]
    (+ for N>1: NCCL all_gather of the keypoint tensors, the only exchange the path has).
Workload = BASELINE.json configs[1]: ViT-B COCO-17 bf16, batch 64 synthetic 256x192 crops per GPU (weak scaling:
crops are independent units, each rank owns its own batch).  Random-init weights of that architecture.
`value` is timed on the device with CUDA events (max over ranks); `e2e` goes through the C-ABI host entry point
(vpb_infer_host) with pinned HOST buffers, H2D + D2H inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

MODELS = {"s": (384, 12, 12), "b": (768, 12, 12), "l": (1024, 24, 16), "h": (1280, 32, 16)}
METRIC = "person-crops/sec ViT-B 256x192 bf16"


def flops_per_crop(D: int, depth: int, heads: int, K: int) -> dict:
    """Algorithmic GEMM/conv flops (2*M*N*K) per crop and kernel class -- SURVEY.md section 8a/8d."""
    T = 192
    f = {
        "gemm_patch_embed": 2 * T * 768 * D,
        "gemm_qkv": depth * 2 * T * D * 3 * D,
        "attention": depth * 2 * 2 * heads * T * T * (D // heads),
        "gemm_proj": depth * 2 * T * D * D,
        "gemm_fc1_gelu": depth * 2 * T * D * 4 * D,
        "gemm_fc2": depth * 2 * T * 4 * D * D,
        "gemm_deconv": 4 * 2 * T * 4 * D * 256 + 4 * 2 * 768 * 1024 * 256,
        "gemm_final_conv": 2 * 3072 * 256 * K,
    }
    f["total"] = sum(f.values())
    # the chained launches (chain.cuh) carry the patch-embed, qkv, proj, fc1 and fc2 GEMMs of the step
    f["gemm_chain"] = f["gemm_patch_embed"] + f["gemm_qkv"] + f["gemm_proj"] + f["gemm_fc1_gelu"] + f["gemm_fc2"]
    return f


def measured_peaks() -> tuple[dict, str]:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh), "measured"
    # fallback stated in /opt/skills/guides/B200_PROFILING.md
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines: list[str] = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()           # exactly the PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ CPU oracle arm
def host_cores() -> int:
    """Cores this process may really use: CPU affinity mask and cgroup v2/v1 CPU quota, not the machine's core count
    (a container that sees 128 CPUs but owns a 16-core quota crawls when torch spawns 128 threads)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as fq, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as fp:
                q, per = int(fq.read()), int(fp.read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return n


DATASET_OF_K = {17: "coco", 25: "coco_25", 133: "wholebody"}


def reference_modules(model: str, K: int, sd_np: dict):
    """The UNMODIFIED reference (`ViTPose(cfg)` from vit_models/model.py + keypoints_from_heatmaps), imported from
    /root/reference or from the copy pip left in baseline/_ref, with the seeded weights loaded strictly -- or None when
    neither is reachable (then the arms below fall back to oracle/torch_ref.py, kind "port")."""
    try:
        import torch

        from oracle import ref_import
        if not ref_import.available() or K not in DATASET_OF_K:
            return None
        ns = ref_import.load()
        net = ns.ViTPose(ns.dyn_model_import(DATASET_OF_K[K], model)).eval()
        net.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd_np.items()}, strict=True)
        return ns, net
    except Exception as exc:                                  # a broken install must not take the bench down
        print(f"[bench] reference import failed, using the port: {exc!r}", file=sys.stderr)
        return None


def oracle_throughput(model: str, K: int, sample_crops: int, steps: int, warmup: int) -> tuple[float, float, int, str]:
    """crops/s of the reference's own CPU path on `sample_crops` crops per step with every host core torch / BLAS will
    use.  kind "reference": the imported reference modules -- ViTPose(cfg).forward in fp32 on one [n,3,256,192] batch, then
    VitInference.postprocess per crop (keypoints_from_heatmaps, easy_ViTPose/inference.py:187-205).  kind "port" (reference
    unreachable): oracle/torch_ref.py (the same torch ops) + the numpy decode restatement."""
    import torch

    from oracle import torch_ref as T
    from oracle import vitpose_oracle as O
    D, depth, heads = MODELS[model]
    cores = host_cores()
    sd_np = O.make_state_dict(D, depth, K, seed=1, peaky=0.1, bumps=True)
    ref = reference_modules(model, K, sd_np)
    sd = T.to_device(sd_np, "cpu", torch.float32)
    x = torch.from_numpy(O.make_crops(sample_crops, seed=2))
    # torchrun pins OMP_NUM_THREADS=1, and containers often see more CPUs than they own: probe a few thread counts on
    # a 2-crop forward and keep the fastest ("all the host threads it can use" = the count that actually helps)
    best_n, best_t = cores, None
    for n in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
        torch.set_num_threads(n)
        with torch.no_grad():
            T.forward(x[:2], sd, depth, heads)
            t0 = time.perf_counter()
            T.forward(x[:2], sd, depth, heads)
            dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_n, best_t = n, dt
    cores = best_n
    torch.set_num_threads(cores)
    org = np.tile(np.array([[192, 256]], np.int32), (sample_crops, 1))

    def one():
        with torch.no_grad():
            if ref is not None:
                from oracle import ref_import
                hm = ref[1](x).numpy()
                return [ref_import.postprocess(ref[0], hm[i:i + 1], int(org[i, 0]), int(org[i, 1])) for i in range(sample_crops)]
            hm = T.forward(x, sd, depth, heads).numpy()
        return O.decode_maps(hm, org, wrap="crop")

    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = time.perf_counter() - t0
    return sample_crops * steps / dt, dt / steps * 1e3, torch.get_num_threads(), ("reference" if ref is not None else "port")


def torch_cuda_eager(model: str, K: int, B: int, dev) -> dict:
    """The target the north star names: the reference's torch-CUDA eager forward (library kernels), restated in
    oracle/torch_ref.py because the reference package cannot travel; fp32 as shipped and .to(bfloat16), forward only."""
    import torch

    from oracle import torch_ref as T
    from oracle import vitpose_oracle as O
    D, depth, heads = MODELS[model]
    sd_np = O.make_state_dict(D, depth, K, seed=1, peaky=0.1, bumps=True)
    ref = reference_modules(model, K, sd_np)
    out = {}
    for name, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        if ref is not None:                                  # ViTPose(cfg).to('cuda')[.to(bfloat16)]: easy_ViTPose/inference.py:156-167
            net = ref[1].to(dev).to(dt)
            fwd = lambda x: net(x)
        else:
            sd = T.to_device(sd_np, dev, dt)
            fwd = lambda x: T.forward(x, sd, depth, heads)
        x = torch.randn((B, 3, 256, 192), device=dev, dtype=dt)
        with torch.no_grad():
            for _ in range(5):
                fwd(x)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(20):
                fwd(x)
            e1.record()
            torch.cuda.synchronize()
        out[name + "_crops_per_s"] = B * 20 / (e0.elapsed_time(e1) / 1e3)
        del x
    out["kind"] = "reference" if ref is not None else "port"
    out["note"] = ("the reference's own ViTPose(cfg) module on the GPU" if ref is not None else "oracle/torch_ref.py restatement") + \
        ": torch eager forward only (no decode), same box, same run; allow_tf32 as torch ships it"
    return out


def bench_frame_path(model, B: int, K: int, steps: int, dev) -> dict:
    """SURVEY.md section 8 rows f1/f2: the reference's whole per-person loop (box pad/clip, crop, pad_image, cv2 resize,
    normalise, model, decode, offset back) as one engine call per frame.  HOST uint8 1080p frames + B boxes in, HOST
    keypoints out, two frames in flight (vpb_submit_frame_host / vpb_wait_host); plus the device time of the
    pre-processing kernel alone and the reference's own CPU pre-processing (cv2) on the same boxes."""
    import torch
    rs = np.random.RandomState(5)
    FH, FW = 1080, 1920
    frames = [torch.from_numpy(rs.randint(0, 256, size=(FH, FW, 3), dtype=np.uint8)).pin_memory() for _ in range(2)]
    w = rs.randint(90, 420, size=B); h = (w * rs.uniform(1.6, 2.6, size=B)).astype(np.int64)
    x0 = rs.randint(0, FW - 100, size=B); y0 = rs.randint(0, FH - 200, size=B)
    boxes = np.ascontiguousarray(np.stack([x0, y0, x0 + w, y0 + h], 1).astype(np.int32))
    hk = [torch.empty((B, K, 3), dtype=torch.float32).pin_memory().numpy() for _ in range(2)]
    hi = [torch.empty((B, K), dtype=torch.int32).pin_memory().numpy() for _ in range(2)]
    fr = [f.numpy() for f in frames]
    for _ in range(3):
        model.infer_frame_host(fr[0], boxes)
    for i in range(3):                                    # warm the pipelined entry (graph capture on its stream, staging slots)
        model.submit_frame_host(fr[i % 2], boxes, hk[i % 2], hi[i % 2], i % 2)
        model.wait_host(i % 2)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    model.submit_frame_host(fr[0], boxes, hk[0], hi[0], 0)
    for i in range(1, steps):
        model.submit_frame_host(fr[i % 2], boxes, hk[i % 2], hi[i % 2], i % 2)
        model.wait_host((i - 1) % 2)
    model.wait_host((steps - 1) % 2)
    dt = time.perf_counter() - t0
    # the pre-processing kernel alone, CUDA events on its stream, frame resident
    d_frame = frames[0].to(dev); d_boxes = torch.from_numpy(boxes).to(dev)
    import ctypes as C

    from easy_vitpose_b200 import _lib
    crops = torch.empty((B, 3, 256, 192), dtype=torch.float32, device=dev)
    org = torch.empty((B, 2), dtype=torch.int32, device=dev); offs = torch.empty((B, 2), dtype=torch.int32, device=dev)
    side = torch.cuda.Stream(dev)

    def pp():
        _lib.check(_lib.lib().vpb_preprocess(C.c_void_p(d_frame.data_ptr()), FH, FW, 0, C.c_void_p(d_boxes.data_ptr()), B, 10,
                                             C.c_void_p(crops.data_ptr()), C.c_void_p(org.data_ptr()), C.c_void_p(offs.data_ptr()),
                                             None, C.c_void_p(side.cuda_stream)))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 50
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        for _ in range(5):
            pp()
        e0.record(side)
        for _ in range(reps):
            pp()
        e1.record(side)
    torch.cuda.synchronize()
    pp_ms = e0.elapsed_time(e1) / reps                 # back-to-back launches on one stream, frame resident in L2/HBM
    out_bytes = B * 3 * 256 * 192 * 4
    # the fused kernel the frame path actually runs (frame -> bf16 patch rows + token-stream seed), engine profiler events
    model.set_option("profile", 1)
    model.profile_collect()
    with torch.cuda.stream(side):
        for _ in range(10):
            model.infer_frame(d_frame, d_boxes)
    torch.cuda.synchronize()
    fused_ms, fused_n = model.profile_collect()["crop_preprocess"]
    model.set_option("profile", 0)
    D = model.embed_dim
    fused_bytes = B * 192 * 768 * 2 + B * 192 * D * 4          # bf16 patch rows + fp32 token-stream seed written
    res = {"workload": f"{FH}x{FW} uint8 RGB frame + {B} person boxes per step, host in / host out",
           "value": B * steps / dt, "unit": "crops/s", "frames_per_s": steps / dt, "steps": steps,
           "api": "vpb_submit_frame_host / vpb_wait_host (C ABI), 2 frames in flight, pinned host buffers",
           "h2d_bytes_per_step": FH * FW * 3 + B * 16, "d2h_bytes_per_step": B * K * 3 * 4 + B * K * 4,
           "preprocess_kernel": {"ms_per_call": pp_ms, "bytes_written": out_bytes, "GBps_written": out_bytes / (pp_ms * 1e-3) / 1e9,
                                 "note": "vpb_preprocess (f32 crops), CUDA events around 50 back-to-back launches"},
           "fused_gather_kernel": {"ms_per_call": fused_ms / max(1, fused_n), "bytes_written": fused_bytes,
                                   "GBps_written": fused_bytes / (fused_ms / max(1, fused_n) * 1e-3) / 1e9,
                                   "note": "frame_to_patch_rows inside vpb_infer_frame: replaces crop_resize_normalise + patch_im2col"}}
    try:
        import cv2
        MEAN, STD = np.array([0.485, 0.456, 0.406]), np.array([0.229, 0.224, 0.225])
        n_cpu = min(B, 32)
        t0 = time.perf_counter()
        for b in boxes[:n_cpu]:
            # what VitInference.inference does per person on the CPU (easy_ViTPose/inference.py:259-265,314-318)
            x0, x1 = np.clip([b[0] - 10, b[2] + 10], 0, FW); y0, y1 = np.clip([b[1] - 10, b[3] + 10], 0, FH)
            crop = fr[0][y0:y1, x0:x1]
            h, w = crop.shape[:2]
            if w / h < 3 / 4:
                pad = int(3 / 4 * h) - w
                crop = np.pad(crop, ((0, 0), (pad // 2, pad - pad // 2), (0, 0)))
            else:
                pad = int(w / (3 / 4)) - h
                crop = np.pad(crop, ((pad // 2, pad - pad // 2), (0, 0), (0, 0)))
            x = cv2.resize(crop, (192, 256), interpolation=cv2.INTER_LINEAR) / 255
            x = ((x - MEAN) / STD).transpose(2, 0, 1)[None].astype(np.float32)
        cdt = time.perf_counter() - t0
        res["cpu_preprocess_reference"] = {"value": n_cpu / cdt, "unit": "crops/s", "cores": 1,
                                           "sample": f"{n_cpu} boxes: numpy crop + pad, cv2.resize, float64 normalise (inference.py:259-265,314-318)"}
    except Exception as exc:                                  # cv2 missing on the box: report, do not fail the bench
        res["cpu_preprocess_reference"] = {"unavailable": repr(exc)}
    return res


def workload_name(model: str, K: int, B: int, streams: int = 0) -> str:
    """config.workload, the same string in both arms."""
    if streams:
        return (f"ViT-{model.upper()} K={K} bf16, one synthetic 1080p video stream per GPU, {streams} frames per step with ragged "
                f"detector crop batches (Poisson(10), 1..{B} crops) (BASELINE configs[4]: ViT-B AP-10k streams)")
    tag = {("b", 17, 64): "BASELINE configs[1]: ViT-B COCO-17, batch 64", ("h", 133, 32): "BASELINE configs[2]: ViT-H wholebody-133, batch 32",
           ("l", 25, 64): "BASELINE configs[3]: ViT-L COCO-25, 512 crops over 8 GPUs = 64 per GPU"}.get((model, K, B))
    return f"ViT-{model.upper()} K={K} bf16, batch={B} synthetic 256x192 crops per GPU" + (f" ({tag})" if tag else "")


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    D, depth, heads = MODELS[args.model]
    sample = args.cpu_sample
    value, ms, cores, kind = oracle_throughput(args.model, args.keypoints, sample, args.steps, args.warmup)
    how = ("UNMODIFIED reference: ViTPose(cfg).forward fp32 + keypoints_from_heatmaps per crop" if kind == "reference"
           else "torch CPU fp32 forward + numpy decode (oracle/ port)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "crops/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.model, args.keypoints, args.batch, args.stream_frames), "batch_per_gpu": args.batch,
                   "global_batch": args.gpus * args.batch,
                   "reference_sample": f"each step = {sample} crops of that workload on the host cores (bounded sample)"},
        "cpu_baseline": {"value": value, "unit": "crops/s", "cores": cores, "kind": kind,
                         "sample": f"{sample} crops/step x {args.steps} steps, {how}"},
        "e2e": {"value": value, "unit": "crops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
CONFIGS = {
    # BASELINE.json configs[1..4] as bench presets (crops per GPU; configs[3] is 512 crops over 8 GPUs = 64 per rank)
    "b17x64": dict(model="b", keypoints=17, batch=64, note="BASELINE configs[1]: ViT-B COCO-17, batch 64"),
    "h133x32": dict(model="h", keypoints=133, batch=32, note="BASELINE configs[2]: ViT-H wholebody-133, batch 32"),
    "l25x64": dict(model="l", keypoints=25, batch=64, note="BASELINE configs[3]: ViT-L COCO-25, 512 crops sharded over 8 GPUs = 64 per GPU"),
    "ap10k-streams": dict(model="b", keypoints=17, batch=32, streams=16,
                          note="BASELINE configs[4]: ViT-B AP-10k (K=17), one synthetic video stream per GPU, ragged detector crop batches"),
}


def stream_workload(rank: int, frames: int, max_n: int):
    """One synthetic video stream: `frames` 1080p uint8 frames, each with its own number of detector boxes
    (Poisson(10) clipped to 1..max_n) of person-like sizes.  Seeded per rank: every GPU owns a different stream."""
    rs = np.random.RandomState(4000 + rank)
    FH, FW = 1080, 1920
    counts = np.clip(rs.poisson(10, size=frames), 1, max_n)
    boxes = []
    for n in counts:
        w = rs.randint(90, 420, size=n); h = (w * rs.uniform(1.6, 2.6, size=n)).astype(np.int64)
        x0 = rs.randint(0, FW - 100, size=n); y0 = rs.randint(0, FH - 200, size=n)
        boxes.append(np.ascontiguousarray(np.stack([x0, y0, x0 + w, y0 + h], 1).astype(np.int32)))
    imgs = [rs.randint(0, 256, size=(FH, FW, 3), dtype=np.uint8) for _ in range(4)]      # 4 distinct frames, rotated
    return imgs, boxes, counts


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each array as out_dir/<name>.npy in float32 / float64.  The inputs and weights are seeded, so two builds run
    with the same arguments can be compared output for output."""
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20, "outputs to dump exceed 64 MB"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_gpu(args) -> None:
    import torch
    import torch.distributed as dist

    from easy_vitpose_b200 import ViTPose, model_cfg
    from easy_vitpose_b200.distributed import ShardPipeline
    from easy_vitpose_b200.synthetic import random_state_dict      # the GPU arm never touches oracle/

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's banner / warnings must not land on stdout next to the JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)

    D, depth, heads = MODELS[args.model]
    K, B = args.keypoints, args.batch
    streams = args.stream_frames
    sd = random_state_dict(args.model, K, seed=1, peaks=True)
    model = ViTPose(model_cfg(args.model, K), max_batch=B)
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}).to(dev)
    del sd

    comm = torch.cuda.Stream(dev) if world > 1 else None
    ev_kp = torch.cuda.Event()
    if not streams:
        # inputs: NBUF different batches resident in HBM, rotated so that consecutive steps never re-read the same crops
        NBUF = 4
        g = torch.Generator(device=dev).manual_seed(1000 + rank)
        crops = [torch.randn((B, 3, 256, 192), generator=g, device=dev, dtype=torch.float32) for _ in range(NBUF)]
        org_wh = torch.tensor([[192, 256]] * B, dtype=torch.int32, device=dev)
        gathered = torch.empty((world * B, K, 3), dtype=torch.float32, device=dev) if world > 1 else None
        crops_per_step = B
        l2_note = (f"inputs rotate over {NBUF} device batches ({NBUF * B * 589824 / 1e6:.0f} MB > 126 MB L2); "
                   "weights + activations touched per step exceed L2 several times over")

        def step(i: int):
            kp, idx = model.infer_crops(crops[i % NBUF], org_wh)
            if world > 1:
                # the path's only exchange: final keypoints, gathered on a side stream so it never sits between two
                # steps of the compute stream (13 KB per rank: pure latency)
                ev_kp.record()
                comm.wait_event(ev_kp)
                with torch.cuda.stream(comm):
                    kp.record_stream(comm)
                    dist.all_gather_into_tensor(gathered, kp)
            return [(kp, idx)]
    else:
        # configs[4]: one video stream per GPU; a step = `streams` consecutive frames, each with its own ragged crop batch,
        # through the frame-level entry point (uint8 frame + boxes resident in HBM -> frame keypoints)
        imgs, boxes, counts = stream_workload(rank, streams, B)
        d_imgs = [torch.from_numpy(im).to(dev) for im in imgs]
        d_boxes = [torch.from_numpy(b).to(dev) for b in boxes]
        crops_per_step = int(counts.sum())
        cps = torch.tensor([crops_per_step], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(cps)                               # whole-job crops per step (streams differ per rank)
        total_crops_per_step = int(cps.item())
        comm = None                                            # a stream's keypoints stay on its GPU: no exchange at all
        l2_note = (f"4 distinct 1080p frames rotated (25 MB), {streams} ragged batches per step "
                   f"({int(counts.min())}..{int(counts.max())} crops, {crops_per_step} per step on rank 0's stream)")

        def step(i: int):
            return [model.infer_frame(d_imgs[(i * streams + f) % 4], d_boxes[f]) for f in range(streams)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()

    # ---- parity inside the bench run: the timed batch size against the engine's own one-crop-at-a-time result
    parity = None
    if not streams:
        kp_full, idx_full = model.infer_crops(crops[0], org_wh)
        pick = sorted({0, B // 2, B - 1})
        same = True
        for j in pick:
            kp1, idx1 = model.infer_crops(crops[0][j:j + 1], org_wh[j:j + 1])
            same = same and bool(torch.equal(kp1[0], kp_full[j])) and bool(torch.equal(idx1[0], idx_full[j]))
        parity = {"batch_equals_single_crop_calls": same, "crops_checked": pick,
                  "note": "keypoints + argmax of crops taken from the timed batch == the same crops run alone (bit-exact)"}
        barrier()

    # ---- timed region 1: K steps back to back, device events, nothing else on the stream -> `value`
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(args.steps - 1):
        step(i)
    last = step(args.steps - 1)
    if comm is not None:
        torch.cuda.current_stream().wait_stream(comm)          # the last gathers are part of the timed work
    ev1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        # (keypoints, argmax) of every call in the last timed step, as the caller received them
        outputs = {"keypoints": torch.cat([kp for kp, _ in last]), "argmax": torch.cat([idx for _, idx in last]).double()}
        if world > 1 and not streams:
            outputs["keypoints_all_ranks"] = gathered
        dump_outputs(args.dump_outputs, {name: t.cpu().numpy() for name, t in outputs.items()})
    ms_total = ev0.elapsed_time(ev1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    job_crops_per_step = total_crops_per_step if streams else world * B
    value = job_crops_per_step * args.steps / (ms_total / 1e3)

    # ---- timed region 2: the same K steps with a CUDA-event pair around every kernel launch (recorded by the engine on
    # the launch stream) -> per-kernel durations for the roofline.  The event records sit between the kernels, so this
    # pass runs without launch overlap and is a little slower than region 1; shares are computed against its own total.
    model.set_option("profile", 1)
    pv0, pv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    pv0.record()
    for i in range(args.steps):
        step(i)
    pv1.record()
    barrier()
    ms_prof_total = pv0.elapsed_time(pv1)
    clocks = sampler.stop() if rank == 0 else None
    prof = model.profile_collect()
    prof_unchained = None
    if prof.get("gemm_chain", (0.0, 0))[1] > 0:
        # the chained launches hide the per-GEMM split: one more profiled pass with one kernel per GEMM / LayerNorm
        # (set_option("chain", 0)) for the per-class table and the attention-GEMM figure the north star asks for
        model.set_option("chain", 0)
        for i in range(3):
            step(i)
        barrier()
        model.profile_collect()
        for i in range(args.steps):
            step(i)
        barrier()
        prof_unchained = model.profile_collect()
        model.set_option("chain", 1)
    model.set_option("profile", 0)

    # ---- end to end with pinned HOST buffers, host->device and device->host copies inside the timed region.
    e_steps = max(5, args.steps // 2)
    h_org = torch.tensor([[192, 256]] * B, dtype=torch.int32).pin_memory()
    e2e_sync_value = None
    frame_latency = None
    if streams:
        # host uint8 frames + boxes in, host frame keypoints out, two frames in flight (vpb_submit_frame_host / vpb_wait_host)
        pin = [torch.from_numpy(im).pin_memory().numpy() for im in imgs]
        hk = [[np.empty((int(c), K, 3), np.float32) for c in counts] for _ in range(2)]
        hi = [[np.empty((int(c), K), np.int32) for c in counts] for _ in range(2)]
        for f in range(min(streams, 3)):
            model.infer_frame_host(pin[f % 4], boxes[f])
        for rep in range(2):                              # every ragged batch size twice through the pipelined entry: graphs captured
            for f in range(streams):
                model.submit_frame_host(pin[f % 4], boxes[f], hk[f % 2][f], hi[f % 2][f], f % 2)
                model.wait_host(f % 2)
        barrier()
        t0 = time.perf_counter()
        n_sub = 0
        for i in range(e_steps):
            for f in range(streams):
                slot = n_sub % 2
                if n_sub >= 2:
                    model.wait_host(slot)
                model.submit_frame_host(pin[(i * streams + f) % 4], boxes[f], hk[slot][f], hi[slot][f], slot)
                n_sub += 1
        model.wait_host(0); model.wait_host(1)
        e_dt = time.perf_counter() - t0
        api = "vpb_submit_frame_host / vpb_wait_host (C ABI), 2 frames in flight, pinned host frames"
        h2d = int(1080 * 1920 * 3 * streams + crops_per_step * 16)
        d2h = int(crops_per_step * K * 16)
        # per-frame latency (SURVEY 8d, config 5): one synchronous call per frame -- host frame + boxes in, H2D, the path, D2H,
        # stream sync, keypoints in host memory -- nothing else in flight
        lat = []
        for i in range(max(3, e_steps // 2)):
            for f in range(streams):
                t1 = time.perf_counter()
                model.infer_frame_host(pin[(i * streams + f) % 4], boxes[f])
                lat.append((time.perf_counter() - t1) * 1e3)
        lat = np.sort(np.asarray(lat))
        frame_latency = {"api": "vpb_infer_frame_host (synchronous, one frame in flight)", "frames": int(lat.size),
                         "mean_ms": float(lat.mean()), "p50_ms": float(lat[lat.size // 2]), "p90_ms": float(lat[int(lat.size * 0.9)]),
                         "p99_ms": float(lat[min(lat.size - 1, int(lat.size * 0.99))]), "max_ms": float(lat[-1])}
    elif world == 1:
        h_crops = [torch.randn((B, 3, 256, 192), dtype=torch.float32).pin_memory() for _ in range(2)]
        h_kp = [torch.empty((B, K, 3), dtype=torch.float32).pin_memory() for _ in range(2)]
        h_idx = [torch.empty((B, K), dtype=torch.int32).pin_memory() for _ in range(2)]
        hc, ho = [t.numpy() for t in h_crops], h_org.numpy()
        hk, hi = [t.numpy() for t in h_kp], [t.numpy() for t in h_idx]
        for _ in range(max(3, args.warmup // 2)):
            model.infer_host(hc[0], ho, hk[0], hi[0])
        barrier()
        t0 = time.perf_counter()
        for _ in range(e_steps):
            model.infer_host(hc[0], ho, hk[0], hi[0])     # synchronous: returns after the D2H copy landed
        torch.cuda.synchronize()
        e2e_sync_value = B * e_steps / (time.perf_counter() - t0)
        barrier()
        for i in range(3):                                # warm the pipelined path itself (its stream's CUDA graph is captured on
            model.submit_host(hc[i % 2], ho, hk[i % 2], hi[i % 2], i % 2)     # the second use after the profiling passes reset it)
            model.wait_host(i % 2)
        barrier()
        t0 = time.perf_counter()
        model.submit_host(hc[0], ho, hk[0], hi[0], 0)
        for i in range(1, e_steps):
            model.submit_host(hc[i % 2], ho, hk[i % 2], hi[i % 2], i % 2)
            model.wait_host((i - 1) % 2)
        model.wait_host((e_steps - 1) % 2)
        e_dt = time.perf_counter() - t0
        api = "vpb_submit_host / vpb_wait_host (C ABI), 2 batches in flight, pinned host buffers"
        h2d, d2h = int(B * 3 * 256 * 192 * 4 + B * 8), int(B * K * 3 * 4 + B * K * 4)
    else:
        # N > 1: this rank's pinned crops -> its engine -> NCCL all_gather of the keypoints on a side stream -> pinned host,
        # two batches in flight per rank (easy_vitpose_b200.distributed.ShardPipeline); no blocking call inside the loop
        # except the wait for the batch submitted two steps earlier
        h_crops = [torch.randn((B, 3, 256, 192), dtype=torch.float32).pin_memory() for _ in range(2)]
        pipe = ShardPipeline(model, B, depth=2)
        for i in range(3):
            pipe.submit(i % 2, h_crops[i % 2], h_org); pipe.wait(i % 2)
        barrier()
        t0 = time.perf_counter()
        pipe.submit(0, h_crops[0], h_org)
        for i in range(1, e_steps):
            pipe.submit(i % 2, h_crops[i % 2], h_org)
            pipe.wait((i - 1) % 2)
        pipe.wait((e_steps - 1) % 2)
        e_dt = time.perf_counter() - t0
        api = ("ShardPipeline: pinned host crops -> engine on the rank's shard -> NCCL all_gather of keypoints (side stream) "
               "-> pinned host, 2 batches in flight per rank")
        h2d, d2h = int(B * 3 * 256 * 192 * 4 + B * 8), int(world * B * K * 3 * 4)
    te = torch.tensor([e_dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = job_crops_per_step * e_steps / float(te[0].item())

    frame_path = None
    if world == 1 and not streams and not args.no_frame_path:
        frame_path = bench_frame_path(model, B, K, max(5, args.steps // 2), dev)

    if rank == 0:
        peaks, peak_src = measured_peaks()
        fl = flops_per_crop(D, depth, heads, K)
        kernels = {}
        for name, (ms, n) in prof.items():
            if n == 0:
                continue
            ent = {"ms_per_step": ms / args.steps, "launches_per_step": n / args.steps, "share": ms / ms_prof_total}
            if name in fl:
                ent["tflops"] = fl[name] * crops_per_step * args.steps / (ms / 1e3) / 1e12
            kernels[name] = ent
        # dominant kernel = the class with the largest share of device time
        dom = max((k for k in kernels if "tflops" in kernels[k]), key=lambda k: kernels[k]["ms_per_step"])
        # denominators: the burst cuBLAS figure when the run saw no power cap (short run at full clocks), the sustained
        # one when sw_power_cap was active during the timed region; both fractions are reported
        capped = bool(clocks and "sw_power_cap" in (clocks.get("reasons") or []))
        peak_burst = float(peaks.get("bf16_tflops", 0.0)) or None
        peak_sust = float(peaks.get("bf16_tflops_sustained", 0.0)) or peak_burst
        peak_tf = peak_sust if capped or peak_burst is None else peak_burst
        traffic = None          # dram__bytes_read+write of the dominant kernel, one ncu --set full capture (profiles/)
        try:
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
                traffic = json.load(fh)["dram_bytes_per_launch"].get(dom) if (args.model, B, bool(streams)) == ("b", 64, False) else None
        except Exception:
            traffic = None
        whole = fl["total"] * job_crops_per_step / world * args.steps / (ms_total / 1e3) / 1e12
        pu = prof_unchained or prof
        att_ms = pu["gemm_qkv"][0] + pu["attention"][0] + pu["gemm_proj"][0]
        kernels_unchained = None
        if prof_unchained is not None:
            kernels_unchained = {name: {"ms_per_step": ms / args.steps, "launches_per_step": n / args.steps,
                                        **({"tflops": fl[name] * crops_per_step * args.steps / (ms / 1e3) / 1e12} if name in fl and ms > 0 else {})}
                                 for name, (ms, n) in prof_unchained.items() if n}
        roofline = {"kernel": dom, "bound": "tensor", "achieved": kernels[dom]["tflops"], "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": kernels[dom]["tflops"] / peak_tf,
                    "peak_source": f"{peak_src} " + ("bf16_tflops_sustained (sw_power_cap active in the timed region)" if peak_tf == peak_sust and capped
                                                     else "bf16_tflops (burst: no power cap seen)"),
                    "frac_of_burst": kernels[dom]["tflops"] / peak_burst if peak_burst else None,
                    "frac_of_sustained": kernels[dom]["tflops"] / peak_sust if peak_sust else None,
                    "traffic": traffic, "traffic_unit": "bytes/launch (ncu --set full, profiles/ncu_traffic.json)",
                    "flops_per_launch": fl[dom] * crops_per_step / max(1.0, kernels[dom]["launches_per_step"]),
                    "whole_step_tflops": whole, "whole_step_frac_of_burst": whole / peak_burst if peak_burst else None,
                    "whole_step_frac_of_sustained": whole / peak_sust if peak_sust else None,
                    "attention_gemm_tflops": (fl["gemm_qkv"] + fl["attention"] + fl["gemm_proj"]) * crops_per_step * args.steps / (att_ms / 1e3) / 1e12}
        # CPU baseline: the reference (or its port) on this box's host cores, bounded sample
        cpu_val, cpu_ms, cores, cpu_kind = (None, None, os.cpu_count(), "port")
        eager = None
        if world == 1 and not args.no_cpu_baseline:
            cpu_val, cpu_ms, cores, cpu_kind = oracle_throughput(args.model, K, args.cpu_sample, 3, 1)
            eager = torch_cuda_eager(args.model, K, B, dev)
        line = {
            "metric": METRIC, "value": value, "unit": "crops/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_name(args.model, K, B, streams),
                       "batch_per_gpu": B, "global_batch": job_crops_per_step, "parallelism": f"dp{world} (crops sharded, weights replicated)",
                       "l2": l2_note, "weights": "random init (seeded), bump pathway so heatmaps have peaks"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "crops/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e_steps, "api": api,
                    "single_call_value": e2e_sync_value, "single_call_api": "vpb_infer_host (H2D, path, D2H, sync per call)"},
            "gpu_launches": (model.kernel_launches(B) * (streams or 1)) * args.steps,
            "frame_latency": frame_latency,
            "roofline": roofline,
            "parity_check": parity,
            "profiled_pass_ms_per_step": ms_prof_total / args.steps,
            "kernels": kernels,
            "kernels_unchained": kernels_unchained,
            "cpu_baseline": None if cpu_val is None else {
                "value": cpu_val, "unit": "crops/s", "cores": cores, "kind": cpu_kind,
                "sample": f"{args.cpu_sample} crops x 3 steps, " + ("UNMODIFIED reference ViTPose(cfg).forward fp32 + keypoints_from_heatmaps per crop"
                                                                    if cpu_kind == "reference" else "torch CPU fp32 forward + numpy decode (oracle/ port)")},
            "torch_cuda_eager": eager,
            "frame_path": frame_path,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="b", choices=list(MODELS))
    ap.add_argument("--keypoints", type=int, default=17)
    ap.add_argument("--batch", type=int, default=64, help="crops per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=16, help="crops per CPU-oracle step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-frame-path", action="store_true", help="skip the frame-level (f1/f2) section of the N=1 line")
    ap.add_argument("--config", default=None, choices=list(CONFIGS), help="BASELINE.json configs[1..4] presets (override --model/--keypoints/--batch)")
    ap.add_argument("--stream-frames", type=int, default=0, help="video-stream mode: frames (ragged crop batches) per step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the keypoints and argmax the last timed step returned to DIR/<name>.npy")
    args = ap.parse_args()
    if args.config:
        c = CONFIGS[args.config]
        args.model, args.keypoints, args.batch = c["model"], c["keypoints"], c["batch"]
        args.stream_frames = c.get("streams", 0)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the GPU arm (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
