#!/usr/bin/env python
"""bench.py — headline benchmark: YOLOv3-416 (80 classes) frames/s at batch 64 per GPU, preprocess -> NMS.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the detection hot path over one batch of synthetic frames per GPU
(u8 frames -> fused normalise + conv stack on tcgen05 -> head decode -> Soft-NMS -> result records).
Frames are independent, so ranks share nothing: no data-path collective (the only torch.distributed calls are
the timing barrier and the max-over-ranks of the elapsed time).

--config selects the workload (BASELINE.json:configs); the default is the one the metric is quoted on:
  headline  full-416-80, batch 64 per GPU, weak scaling                         (metric line)
  rsu       rsu-416-9, batch 64 per GPU (config 3)
  608       full-608-80, 256 frames sharded over the N GPUs, strong scaling      (config 4)
  serve     full:80 + rsu:9 co-resident on every GPU, 64 decoded-RGB streams through the in-process dispatcher,
            end-to-end frames/s and latency distribution                       (config 5; own JSON shape)
  tiny-cpu  tiny-416-80 batch 1 on the reference CPU path: p50/p90 + stage split (config 1; CPU only)

JSON keys beyond the base contract:
  value         frames/s with the frames already resident in HBM (CUDA events on the launching stream)
  e2e           the same through the C ABI with PINNED HOST frames in and result records out: H2D + D2H inside
                the timed region (fd_submit / fd_collect, two batches in flight; the synchronous fd_detect figure
                is reported next to it)
  roofline      conv stack (tensor bound): algorithmic conv FLOPs per step / device time of fd_forward inside the
                timed steps, against the measured cuBLAS bf16 BURST peak (MEASURED_PEAKS.json); the sustained-peak
                fraction is an extra key
  roofline_pre / roofline_post   the HBM-bound kernels either side of the conv stack, from this run's CUDA events
  parity_in_run two frames of the first timed batch checked against the CPU oracle inside this run
  cpu_baseline  the oracle port of the reference path (torch-CPU fp32 graph executor standing in for ONNX
                Runtime's CPU EP, which is not installable here + the reference's Python pre/post restated),
                timed on this box's host cores on a bounded sample of the same workload (rank 0, N=1 only)
--impl reference times that same CPU path as its own arm.

--dump-outputs DIR (b200 arm of headline / rsu / 608, rank 0) writes what the last timed step computed as
DIR/<name>.npy: the detection records of every frame of the step, one float64 array per record field (det_<field>[frame,
slot], frames in the step's order, slots past det_count zeroed), and the fp32 head tensors of a fixed seeded sample of
those frames (head<i>[k] belongs to frame head_frames[k]).  Model and frames come from fixed seeds, so two builds run
with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

THRESHOLD = 0.1
MAX_DET = 256

WORKLOADS = {
    # name: arch, classes, size, frames per GPU (None: sharded), model seed, scaling
    "headline": dict(arch="full", classes=80, size=416, batch=64, seed=2, scaling="weak"),
    "rsu": dict(arch="rsu", classes=9, size=416, batch=64, seed=3, scaling="weak"),
    "608": dict(arch="full", classes=80, size=608, batch=None, total=256, seed=2, scaling="strong"),
}


def workload_name(w, world):
    if w.get("batch"):
        return f"yolov3-{w['arch']}-{w['size']}x{w['size']}-{w['classes']}cls-bs{w['batch']}-per-gpu"
    return f"yolov3-{w['arch']}-{w['size']}x{w['size']}-{w['classes']}cls-{w['total']}-frames-sharded"


def bench_config(w, world):
    """The `config` object — identical in the b200 and the reference arm (the driver compares them)."""
    return {"workload": workload_name(w, world), "threshold": THRESHOLD,
            "weights": f"random-init (seed {w['seed']}), BatchNorm folded at load",
            "frames": "64 distinct synthetic frames per batch (fastdet_b200.modelgen.synthetic_frame), 4 batches rotated",
            "stages": "u8 frames -> normalise + first conv -> conv stack -> head decode -> Soft-NMS -> records",
            "l2": "inputs larger than L2: 4 x 33 MB frame sets rotate and ~2.5 GB of activations stream through the 126 MB L2 per step; no explicit flush",
            "parallelism": f"frame-sharded x{world}, no collective"}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fp:
            p = json.load(fp)
        return {"bf16": float(p["bf16_tflops"]), "bf16_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                "hbm": float(p["hbm_gbs"]), "source": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"bf16": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.lines = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        rows = [l.split(", ") for (t, l) in self.lines if t0 - 0.1 <= t <= t1 + 0.3] or [l.split(", ") for (_, l) in self.lines]
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); smax.append(float(r[1])); power.append(float(r[2]))
                for name, v in zip(names, r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def make_frames(first_seed: int, n: int, size: int) -> np.ndarray:
    """n DISTINCT synthetic frames (seeds first_seed .. first_seed + n - 1)."""
    from fastdet_b200 import modelgen
    return np.stack([modelgen.synthetic_frame(first_seed + i, size) for i in range(n)])


# ---------------------------------------------------------------------------------------------- CPU arm
def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every core the process may run on."""
    import torch
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    torch.set_num_threads(max(1, n))
    return torch.get_num_threads()


class CpuPath:
    """The reference path on host cores: per frame normalise -> graph (torch-CPU fp32, all threads) -> decode ->
    Soft-NMS, one frame per call exactly like ONNXDetector.perform (batch 1; reference server/detector.py:126-146)."""

    def __init__(self, onnx_bytes, classes, size):
        from oracle import ref_graph
        self.threads = use_all_host_threads()
        self.sess = ref_graph.OrtSubstituteSession(onnx_bytes)
        self.classes, self.size = classes, size
        self.split = {"normalise": 0.0, "model_run": 0.0, "decode": 0.0, "soft_nms": 0.0}
        self.calls = 0

    def perform(self, frame):
        from oracle import ref_post
        t0 = time.perf_counter()
        a = ref_post.normalise(frame)
        t1 = time.perf_counter()
        outs = self.sess.run(None, {"input": a})
        t2 = time.perf_counter()
        cands, first = [], 0
        for anchors, out in zip(ref_post.ANCHORS[len(outs)], outs):
            m = np.ascontiguousarray(out[0].transpose(1, 2, 0))
            cands.extend(ref_post.decode_head(anchors, m, self.classes, (self.size, self.size), THRESHOLD, first))
            first += m.shape[0] * m.shape[1] * 3
        t3 = time.perf_counter()
        kept = ref_post.soft_nms(cands, THRESHOLD)
        t4 = time.perf_counter()
        for k, v in zip(self.split, (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
            self.split[k] += v
        self.calls += 1
        return kept

    def split_ms(self):
        return {k: round(v / max(self.calls, 1) * 1e3, 2) for k, v in self.split.items()}


def cpu_reference_fps(onnx_bytes, w, frames, budget_s, min_frames=2):
    cpu = CpuPath(onnx_bytes, w["classes"], w["size"])
    cpu.perform(frames[0])  # warm-up (thread pool, oneDNN primitive cache)
    cpu.split = {k: 0.0 for k in cpu.split}
    cpu.calls = 0
    done = 0
    t_start = time.perf_counter()
    while True:
        cpu.perform(frames[done % len(frames)])
        done += 1
        if done >= min_frames and time.perf_counter() - t_start >= budget_s:
            break
    total = time.perf_counter() - t_start
    return done / total, done, total, cpu.split_ms(), cpu.threads


def run_reference(args):
    rank, world, local = dist_env()
    if rank != 0:
        return 0
    from fastdet_b200 import modelgen
    w = WORKLOADS[args.config]
    onnx_bytes = modelgen.build_onnx(w["arch"], w["classes"], w["size"], w["seed"])
    frames = make_frames(100, 16, w["size"])  # 16 distinct frames of the workload's first batch
    per_step = 2  # bounded sample: 2 frames of the workload per step
    cpu = CpuPath(onnx_bytes, w["classes"], w["size"])

    def step(i):
        for j in range(per_step):
            cpu.perform(frames[(i * per_step + j) % len(frames)])

    for i in range(max(args.warmup, 1)):
        step(i)
    cpu.split = {k: 0.0 for k in cpu.split}
    cpu.calls = 0
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(args.warmup + i)
    dt = time.perf_counter() - t0
    fps = args.steps * per_step / dt
    sample = (f"{per_step} frames/step x {args.steps} steps over 16 distinct frames of the workload, batch 1 per call like "
              f"ONNXDetector.perform; rank 0 only")
    line = {
        "impl": "reference", "metric": "frames_per_second", "value": round(fps, 3), "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True,
        "scaling": w["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(w, max(world, args.gpus)),
        "reference_arm": "oracle port on host CPU: torch-CPU fp32 graph executor in place of onnxruntime's CPU EP (not installable in this "
                         "image) + the reference's pre/post-processing restated (oracle/)",
        "cpu_baseline": {"value": round(fps, 3), "unit": "frames/s", "cores": cpu.threads, "kind": "port", "sample": sample,
                         "host_cpus": os.cpu_count(), "ms_per_frame_split": cpu.split_ms()},
        "e2e": {"value": round(fps, 3), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def run_tiny_cpu(args):
    """BASELINE config 1: YOLOv3-tiny 416 (80 classes), batch 1, on the reference CPU path; dog.jpg (the reference's
    testdata fixture, committed as tests/golden/ref_images.npz) and a dog-shaped synthetic frame; 20 warm-up + --steps
    timed calls (200 unless given); p50 / p90 and the stage split."""
    rank, _, _ = dist_env()
    if rank != 0:
        return 0
    import io

    from PIL import Image

    from fastdet_b200 import modelgen
    onnx_bytes = modelgen.build_onnx("tiny", 80, 416, 1)
    cpu = CpuPath(onnx_bytes, 80, 416)
    payloads = {}
    try:
        z = np.load(os.path.join(ROOT, "tests", "golden", "ref_images.npz"))
        payloads["dog.jpg"] = z["dog_jpg"].tobytes()
    except Exception:
        pass
    buf = io.BytesIO()
    Image.fromarray(modelgen.synthetic_frame(0, 416), "RGB").save(buf, format="JPEG", quality=90)
    payloads["synthetic q90"] = buf.getvalue()
    out = {}
    calls = args.steps
    for name, data in payloads.items():
        lat, dec = [], []
        for i in range(20 + calls):
            t0 = time.perf_counter()
            img = Image.open(io.BytesIO(data))  # reference server/detector.py:128-130
            assert img.size == (416, 416)
            frame = np.array(img)
            t1 = time.perf_counter()
            if i == 20:
                cpu.split = {k: 0.0 for k in cpu.split}
                cpu.calls = 0
            cpu.perform(frame)
            if i >= 20:
                lat.append((time.perf_counter() - t0) * 1e3)
                dec.append((t1 - t0) * 1e3)
        out[name] = {"p50_ms": round(float(np.percentile(lat, 50)), 3), "p90_ms": round(float(np.percentile(lat, 90)), 3),
                     "calls": calls, "split_ms": dict(decode_image=round(float(np.mean(dec)), 3), **cpu.split_ms())}
    p50 = out[next(iter(out))]["p50_ms"]
    print(json.dumps({"impl": "reference", "metric": "latency_ms_p50", "value": p50, "unit": "ms", "n_gpus": 0, "steps": calls, "warmup": 20,
                      "higher_is_better": False, "dtype": "f32", "data": "dog.jpg + synthetic",
                      "config": {"workload": "yolov3-tiny-416x416-80cls-bs1 on the reference CPU path (BASELINE config 1)"},
                      "cpu_baseline": {"kind": "port", "cores": cpu.threads, "host_cpus": os.cpu_count(),
                                       "note": "torch-CPU fp32 stands in for onnxruntime's CPU EP (not installable here)"},
                      "frames": out}))
    return 0


# ---------------------------------------------------------------------------------------------- GPU arm
def jpeg_arm(model, frames, n, steps):
    """The same batches entering as JPEG payloads, the way the reference's perform(data) receives them
    (server/detector.py:128-133): fd_submit_jpeg / fd_collect, Huffman decode on the library's host threads inside the
    timed region, IDCT + upsampling + colour conversion on the device.  Reported next to the reference's own decode
    step (PIL, one frame per call, one core)."""
    import io

    import torch
    from PIL import Image
    datas = []
    for f in frames[:16]:
        buf = io.BytesIO()
        Image.fromarray(np.ascontiguousarray(f)).save(buf, "JPEG", quality=75)  # PIL default 4:2:0
        datas.append(buf.getvalue())
    batch = [datas[i % len(datas)] for i in range(n)]
    t0 = time.perf_counter()
    decoded = [np.array(Image.open(io.BytesIO(d))) for d in batch[:16]]
    pil_ms = (time.perf_counter() - t0) / 16 * 1e3
    exact = bool(np.array_equal(model.decode_jpeg(batch[:8]), np.stack(decoded[:8])))

    def run(k):
        model.submit_jpeg(0, batch, THRESHOLD, max_det=MAX_DET)
        for i in range(1, k):
            model.submit_jpeg(i % 2, batch, THRESHOLD, max_det=MAX_DET)
            model.collect((i - 1) % 2)
        model.collect((k - 1) % 2)

    run(3)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    run(steps)
    torch.cuda.synchronize()
    secs = time.perf_counter() - t0
    lat = []
    for i in range(120):
        t0 = time.perf_counter()
        model.detect_jpeg(batch[:1], THRESHOLD, max_det=MAX_DET)
        if i >= 20:
            lat.append((time.perf_counter() - t0) * 1e3)
    return {"value": round(n * steps / secs, 1), "unit": "frames/s",
            "api": "fd_submit_jpeg / fd_collect: JPEG bytes in (quality 75, 4:2:0), Huffman decode on the host pool inside the timed region, "
                   "IDCT + fancy upsampling + YCbCr->RGB on the device, records out",
            "jpeg_kb_per_frame": round(sum(len(d) for d in batch) / n / 1024, 1), "host_threads": os.cpu_count(),
            "pixels_bit_exact_vs_pillow": exact, "reference_decode_ms_per_frame_one_core": round(pil_ms, 3),
            "bs1_latency_ms_p50": round(float(np.percentile(lat, 50)), 4)}


def parity_in_run(model, onnx_bytes, w, frames, n, sp):
    """Two frames of the batch the timed region starts with, through the production execution state (batch n), against
    the CPU oracle: raw heads within 2e-2 * max|ref| (fp32 oracle) and the solid detections found at the same anchor
    boxes with the same classes."""
    from oracle import ref_graph, ref_post
    size, nc = w["size"], w["classes"]
    model.preprocess(frames, n, (size, size))
    model.forward(n)
    heads = model.heads(n)
    model.postprocess(n, THRESHOLD, max_det=MAX_DET)
    dets, counts, _ = model.fetch(n)
    exe = ref_graph.GraphExecutor(onnx_bytes)
    out = {"frames": [0, n // 2 + 5], "head_err_over_max_ref": [], "solid_reference_detections": 0, "found_same_box_and_class": 0}
    for f in out["frames"]:
        ref = exe.run(ref_post.normalise(frames[f]))
        out["head_err_over_max_ref"].append([round(float(np.abs(g[f] - r[0]).max() / np.abs(r).max()), 5) for g, r in zip(heads, ref)])
        want, idx, decayed = ref_post.detect_from_heads(ref, 0, nc, (size, size), THRESHOLD)
        got = {int(d["box"]): int(d["klass"]) for d in dets[f, :counts[f]]}
        for box, r, s in zip(idx, want, decayed):
            if min(r[1], s) >= THRESHOLD + 2e-2:
                out["solid_reference_detections"] += 1
                out["found_same_box_and_class"] += int(got.get(box) == r[0])
    worst = max(max(e) for e in out["head_err_over_max_ref"])
    flips_allowed = max(1, out["solid_reference_detections"] // 40)  # Soft-NMS near-tie flips: one per 40 solid detections (at least one)
    out["ok"] = bool(worst <= 2e-2 and out["found_same_box_and_class"] >= out["solid_reference_detections"] - flips_allowed)
    out["bound"] = ("heads: max|gpu-ref| <= 2e-2 * max|ref| vs the fp32 oracle; detections clearing the threshold by 2e-2 at the same anchor box and class "
                    "(Soft-NMS near-tie flips tolerated: one per 40 such detections, here %d; the GPU tests decide each such case by nudging the oracle's own scores)" % flips_allowed)
    return out


DUMP_HEAD_FRAMES = 4  # full head maps of 4 frames: 14.5 MB at 416 x 416, 31 MB at 608 x 608 (80 classes)
DUMP_LIMIT_BYTES = 64 << 20


def last_step_outputs(model, n, batches, run_batch, sp):
    """--dump-outputs: the records fd_fetch returns for every frame of the last timed step, and the heads of a seeded
    sample of those frames.  The model's buffers hold only the batch it ran last; the step's earlier batches (608: four
    batches of 64 frames per GPU) are run again with run_batch(b) from the same inputs, which the deterministic path
    turns into the same outputs."""
    from fastdet_b200 import _native
    frames = np.sort(np.random.default_rng(0).choice(n * batches, min(n * batches, DUMP_HEAD_FRAMES), replace=False))
    got = {}
    for b in [batches - 1] + list(range(batches - 1)):  # the last batch first, while it is still in the buffers
        if b != batches - 1:
            run_batch(b)
        dets, counts, total = model.fetch(n, stream=sp)
        mine = frames[(frames >= b * n) & (frames < (b + 1) * n)] - b * n
        got[b] = (dets, counts, total, [h[mine] for h in model.heads(n)] if len(mine) else [])
    dets, counts, total = (np.concatenate([got[b][k] for b in range(batches)]) for k in range(3))
    valid = np.arange(dets.shape[1])[None, :] < counts[:, None]
    out = {"det_count": counts.astype(np.float64), "det_total": total.astype(np.float64)}
    for field in _native.DET_DTYPE.names:
        out["det_" + field] = np.where(valid, dets[field], 0).astype(np.float64)
    out["head_frames"] = frames.astype(np.float64)
    for i in range(len(model.head_shapes)):
        out[f"head{i}"] = np.concatenate([got[b][3][i] for b in range(batches) if got[b][3]])
    size = sum(a.nbytes for a in out.values())
    assert size <= DUMP_LIMIT_BYTES, f"--dump-outputs would write {size} bytes"
    return out


def write_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_b200(args):
    import torch
    from fastdet_b200 import _native, modelgen

    rank, world, local = dist_env()
    if world != args.gpus and world > 1:
        print(f"warning: WORLD_SIZE={world} but --gpus {args.gpus}", file=sys.stderr)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    use_dist = world > 1
    if use_dist:
        import torch.distributed as dist
        # NCCL announces its version on stdout when the communicator comes up; the contract is ONE JSON line on
        # stdout, so stdout is pointed at stderr while the process group initialises and runs its first collective.
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    peaks = load_peaks()

    w = WORKLOADS[args.config]
    size, classes = w["size"], w["classes"]
    onnx_bytes = modelgen.build_onnx(w["arch"], classes, size, w["seed"])
    model = _native.Model(onnx_bytes, classes, (size, size), device=local)
    info = model.info
    if w.get("batch"):
        n, batches_per_step = w["batch"], 1
    else:  # a fixed total sharded over the ranks (strong scaling), each rank's shard run in batches of at most 64
        shard = w["total"] // world
        n = min(shard, 64)
        batches_per_step = shard // n
    # four different input sets of n distinct frames each, rotated: 4 x 33 MB of u8 (416) > 126 MB L2 together with the
    # 124 MB of weights; the per-step activation traffic (GBs) flushes L2 many times over anyway.
    sets = [make_frames(10000 * rank + 100 + n * k, n, size) for k in range(4)]
    dev_sets = [torch.from_numpy(s).cuda() for s in sets]
    pin_sets = [torch.from_numpy(s).pin_memory() for s in sets]
    # a dedicated non-default stream: handle 0 would select the model's own internal stream (C ABI: NULL = own stream)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    assert sp != 0

    def run_batch(i, b, ev=None):
        d = dev_sets[(i * batches_per_step + b) % 4]
        model.preprocess(d.data_ptr(), n, (size, size), on_device=True, stream=sp)
        if ev:
            ev[3 * b].record(stream)
        model.forward(n, stream=sp)
        if ev:
            ev[3 * b + 1].record(stream)
        model.postprocess(n, THRESHOLD, max_det=MAX_DET, stream=sp)
        if ev:
            ev[3 * b + 2].record(stream)

    def step_device(i, ev=None):
        for b in range(batches_per_step):
            run_batch(i, b, ev)

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None  # started early: nvidia-smi needs a moment to begin reporting
    parity = parity_in_run(model, onnx_bytes, w, sets[0], n, sp) if rank == 0 and not args.no_parity else None
    for i in range(max(args.warmup, 3)):
        step_device(i)
    torch.cuda.synchronize()
    dets, counts, total = model.fetch(n, stream=sp)
    det_per_frame = float(np.mean(total))

    # ---- timed region 1: device-resident frames, K steps, CUDA events on the launching stream
    step_events = [[torch.cuda.Event(enable_timing=True) for _ in range(3 * batches_per_step)] for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    e0.record(stream)
    for i in range(args.steps):
        step_device(i, step_events[i])
    e1.record(stream)
    barrier()
    t_wall1 = time.time()
    elapsed_ms = e0.elapsed_time(e1)
    fwd_ms = float(np.mean([ev[3 * b].elapsed_time(ev[3 * b + 1]) for ev in step_events for b in range(batches_per_step)]))
    post_ms = float(np.mean([ev[3 * b + 1].elapsed_time(ev[3 * b + 2]) for ev in step_events for b in range(batches_per_step)]))
    # read back before the regions below reuse the model's buffers
    if args.dump_outputs and rank == 0:
        dumped = last_step_outputs(model, n, batches_per_step, lambda b: run_batch(args.steps - 1, b), sp)
    else:
        dumped = None

    # ---- timed region 2: end to end through the synchronous C-ABI call with pinned host frames
    out = np.zeros((n, MAX_DET), _native.DET_DTYPE)
    cnt = np.zeros(n, np.int32)
    lib = _native.lib()
    import ctypes as C

    def step_e2e(i):
        for b in range(batches_per_step):
            p = pin_sets[(i * batches_per_step + b) % 4]
            rc = lib.fd_detect(model._h, C.c_void_p(p.data_ptr()), n, size, size, 0, 0, THRESHOLD, MAX_DET,
                               out.ctypes.data_as(C.c_void_p), cnt.ctypes.data_as(C.c_void_p))
            if rc:
                raise RuntimeError(lib.fd_last_error().decode())

    for i in range(3):
        step_e2e(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step_e2e(i)
    torch.cuda.synchronize()
    e2e_sync_s = time.perf_counter() - t0
    barrier()

    # ---- timed region 3: the same batches through the pipelined pair fd_submit / fd_collect (two slots: the
    # pinned-host -> device copy of batch i+1 overlaps the compute of batch i; every batch's records are read back)
    tot = np.zeros(n, np.int32)

    def submit(i):
        p = pin_sets[i % 4]
        rc = lib.fd_submit(model._h, i % 2, C.c_void_p(p.data_ptr()), n, size, size, 0, 0, THRESHOLD, MAX_DET)
        if rc:
            raise RuntimeError(lib.fd_last_error().decode())

    def collect(i):
        rc = lib.fd_collect(model._h, i % 2, out.ctypes.data_as(C.c_void_p), cnt.ctypes.data_as(C.c_void_p),
                            tot.ctypes.data_as(C.c_void_p))
        if rc:
            raise RuntimeError(lib.fd_last_error().decode())

    def run_pipelined(k):
        submit(0)
        for i in range(1, k):
            submit(i)
            collect(i - 1)
        collect(k - 1)

    run_pipelined(3)
    barrier()
    t0 = time.perf_counter()
    run_pipelined(args.steps * batches_per_step)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    clocks = sampler.stop(t_wall0, time.time()) if sampler else None

    if use_dist:
        t = torch.tensor([elapsed_ms, e2e_s * 1e3, fwd_ms, e2e_sync_s * 1e3, post_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms, e2e_ms, fwd_ms, e2e_sync_ms, post_ms = (float(v) for v in t.tolist())
    else:
        e2e_ms, e2e_sync_ms = e2e_s * 1e3, e2e_sync_s * 1e3

    line = None
    if rank == 0:
        frames_step = n * batches_per_step
        frames_total = world * frames_step * args.steps
        value = frames_total / (elapsed_ms * 1e-3)
        e2e = frames_total / (e2e_ms * 1e-3)
        flops_batch = info.conv_flops_per_frame * n
        achieved = flops_batch / (fwd_ms * 1e-3) * 1e-12
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as fp:
                tj = json.load(fp)
            if args.config == "headline":
                traffic = tj.get("conv_stack_dram_bytes_per_step_bs64")
                traffic_src = "profiles/roofline_traffic.json: ncu dram__bytes_read+write.sum over the conv launches of one step (committed capture " + str(tj.get("source", "")) + ", not this run)"
        except Exception:
            pass
        # the HBM-bound kernels either side of the conv stack, timed in this run
        layer_ms = model.time_layers(n, 10)
        px = n * size * size
        L0 = model.layers()[0]
        exec_rows = model.exec_info(n)
        stem = exec_rows[0]["kernel_name"] == "fused_next"  # conv_stem_kernel: the first convolution runs inside the second one's kernel
        if stem:
            L1 = model.layers()[1]
            pre_bytes = px * 3 + n * L1["h"] * L1["w"] * L1["c"] * 2  # u8 frames in + the SECOND convolution's bf16 output out
            pre_ms = float(layer_ms[1])
            pre_kernel = ("conv_stem_kernel = /255 normalise + first conv (3->32) + second conv (32->64, stride 2) in one kernel: u8 frames in, "
                          "bf16 NHWC of the half-size map out; the first conv's activation (64 B/pixel) stays in shared memory. MMA-issue bound, not HBM bound: "
                          "as two kernels the same work moved %d MB" % ((px * 3 + 2 * px * L0["c"] * 2 + n * L1["h"] * L1["w"] * L1["c"] * 2) // 1000000))
        else:
            pre_bytes = px * 3 + px * L0["c"] * 2  # u8 frame in + bf16 first-conv output out (normalisation fused: no f32 tensor)
            pre_ms = float(layer_ms[0])
            pre_kernel = "conv0_ws_kernel = /255 normalise + layout + first conv fused: u8 frames in (3 B/pixel), bf16 NHWC out"
        pre_gbs = pre_bytes / (pre_ms * 1e-3) * 1e-9
        head_bytes = n * sum(c * h * ww for (c, h, ww) in model.head_shapes) * 4
        post_gbs = head_bytes / (post_ms * 1e-3) * 1e-9
        launches_per_batch = sum(e["launches"] for e in exec_rows) + 2  # conv stack (chunked layers launch once per chunk) + decode + Soft-NMS
        chunked = sorted({(e["chunk_frames"], e["launches"]) for e in exec_rows if e["launches"] > 1})
        line = {
            "metric": "frames_per_second", "value": round(value, 1), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": round(elapsed_ms / args.steps, 4), "higher_is_better": True, "scaling": w["scaling"],
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": bench_config(w, world),
            "frames_per_step_per_gpu": frames_step, "detections_per_frame": round(det_per_frame, 1),
            "e2e": {"value": round(e2e, 1), "unit": "frames/s", "h2d_bytes_per_step": int(frames_step * size * size * 3),
                    "d2h_bytes_per_step": int(frames_step * MAX_DET * 48 + 2 * 4 * frames_step),
                    "api": "fd_submit / fd_collect (C ABI), pinned host frames, two batches in flight; every batch copied in and its records read back",
                    "synchronous_fd_detect": round(frames_total / (e2e_sync_ms * 1e-3), 1)},
            "gpu_launches": int(world * args.steps * batches_per_step * launches_per_batch),
            "roofline": {"bound": "tensor", "achieved": round(achieved, 1), "peak": peaks["bf16"], "unit": "TFLOP/s",
                         "frac": round(achieved / peaks["bf16"], 4), "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "conv stack (conv_tc_kernel / conv_halo_kernel / conv_stem_kernel, all tcgen05/TMEM), timed as fd_forward inside the timed steps",
                         "launches_per_batch": launches_per_batch, "l2_resident_chunks": [{"frames": c, "launches_per_layer": k} for c, k in chunked],
                         "peak_kind": "bf16_tflops (burst: the timed region is well under 1 s of tensor work), " + peaks["source"],
                         "frac_of_sustained_peak": round(achieved / peaks["bf16_sustained"], 4), "peak_sustained": peaks["bf16_sustained"],
                         "forward_ms_per_batch": round(fwd_ms, 4), "flops_per_batch": flops_batch},
            "roofline_pre": {"bound": "hbm", "achieved": round(pre_gbs, 1), "peak": peaks["hbm"], "unit": "GB/s", "frac": round(pre_gbs / peaks["hbm"], 4),
                             "traffic": None, "kernel": pre_kernel,
                             "bytes_per_launch": int(pre_bytes), "ms": round(pre_ms, 4),
                             "how": "fd_time_layers in this run: CUDA events around 10 back-to-back launches of the kernel alone (its output per launch is larger than L2)"},
            "roofline_post": {"bound": "hbm", "achieved": round(post_gbs, 1), "peak": peaks["hbm"], "unit": "GB/s", "frac": round(post_gbs / peaks["hbm"], 4),
                              "traffic": None, "kernel": "decode_kernel + soft_nms_kernel (+ record copy-out)", "bytes_per_launch": int(head_bytes),
                              "ms": round(post_ms, 4),
                              "how": "CUDA events inside the timed steps; algorithmic bytes = fp32 head elements x 4 (SURVEY 8d). The pair is latency-bound "
                                     "(sequential Soft-NMS arg-max), not bandwidth-bound: decode touches only the objectness sectors unless a box passes"},
            "parity_in_run": parity,
            "clocks": clocks,
        }
    # ---- reported CPU baseline + bs1 latency (rank 0, N=1 only)
    if rank == 0 and world == 1 and not args.quick:
        fps, done, secs, split, cores = cpu_reference_fps(onnx_bytes, w, sets[0][:16], budget_s=args.cpu_seconds)
        line["cpu_baseline"] = {"value": round(fps, 3), "unit": "frames/s", "cores": cores, "kind": "port",
                                "sample": f"{done} calls over 16 distinct frames of the same workload in {secs:.1f} s, batch 1 per call like ONNXDetector.perform",
                                "ms_per_frame_split": split, "host_cpus": os.cpu_count(),
                                "note": "oracle port: torch-CPU fp32 stands in for onnxruntime's CPU EP (not installable here)"}
        lat, lat_dev = [], []
        one = pin_sets[0][:1].contiguous().pin_memory()
        o1 = np.zeros((1, MAX_DET), _native.DET_DTYPE)
        c1 = np.zeros(1, np.int32)
        for i in range(1020):
            t0 = time.perf_counter()
            lib.fd_detect(model._h, C.c_void_p(one.data_ptr()), 1, size, size, 0, 0, THRESHOLD, MAX_DET,
                          o1.ctypes.data_as(C.c_void_p), c1.ctypes.data_as(C.c_void_p))
            if i >= 20:
                lat.append((time.perf_counter() - t0) * 1e3)
        d1 = dev_sets[0][:1].contiguous()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(220):
            ea.record(stream)
            model.preprocess(d1.data_ptr(), 1, (size, size), on_device=True, stream=sp)
            model.forward(1, stream=sp)
            model.postprocess(1, THRESHOLD, max_det=MAX_DET, stream=sp)
            eb.record(stream)
            torch.cuda.synchronize()
            if i >= 20:
                lat_dev.append(ea.elapsed_time(eb))
        line["bs1_latency_ms"] = {"p50": round(float(np.percentile(lat, 50)), 4), "p90": round(float(np.percentile(lat, 90)), 4),
                                  "p99": round(float(np.percentile(lat, 99)), 4),
                                  "device_only_p50": round(float(np.percentile(lat_dev, 50)), 4),
                                  "what": "fd_detect, 1 pinned host frame in, records out (H2D + D2H included), 1000 calls, host wall clock; "
                                          "device_only = CUDA events around preprocess(device frame) + forward + postprocess, 200 calls"}
        line["e2e"]["from_jpeg"] = jpeg_arm(model, sets[0], n, args.steps)
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    if rank == 0:
        print(json.dumps(line))
    if use_dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 100; 200 calls for --config tiny-cpu)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="headline", choices=sorted(WORKLOADS) + ["serve", "tiny-cpu"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="time budget of the reported CPU baseline sample")
    ap.add_argument("--quick", action="store_true", help="skip the CPU baseline and the bs1 latency loop (profiling runs)")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run oracle check (profiling runs)")
    ap.add_argument("--seconds", type=float, default=20.0, help="--config serve: length of the measured run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the records of every frame of the last timed step and "
                                                           "the heads of a seeded sample of them as DIR/<name>.npy")
    args = ap.parse_args()
    if args.config == "serve" and args.steps is not None:
        ap.error("--config serve runs for --seconds, not a number of steps")
    if args.steps is None:
        args.steps = 200 if args.config == "tiny-cpu" else 100
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config not in WORKLOADS):
        ap.error("--dump-outputs applies to the b200 arm of " + " / ".join(WORKLOADS))
    if args.config == "tiny-cpu":
        return run_tiny_cpu(args)
    if args.config == "serve":
        from tools import serve_bench
        return serve_bench.main_from_bench(args)
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
