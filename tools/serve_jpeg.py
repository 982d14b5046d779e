#!/usr/bin/env python
"""JPEG requests on the multi-GPU dispatcher: full:80 + rsu:9 co-resident on every visible GPU, N Python caller threads
each sending its next JPEG payload through the drop-in object (``srv.detector(model, stream).perform(data, threshold)``)
as soon as its previous result is back.  Two routes, alternated in one process:

  pil     the route before lanes took JPEG payloads: PIL decode in the caller's thread, then perform_records (RGB batch)
  device  DetectServer.detector(...).perform: the caller entropy-decodes into the lane's JPEG batch, IDCT + colour on the GPU

Thresholds are 0.3 for full and 0.1 for rsu; in the `mixed` variant half of each model's streams use the other model's
threshold (an RGB batch holds one threshold, a JPEG batch any number).  Reports frames/s, latency p50 / p99, mean batch
and host CPU seconds per frame (user + system of this process), with the GPU's name and power limit.

    python tools/serve_jpeg.py [--streams 64,256] [--seconds 5] [--rounds 2] [--out FILE]
"""
import argparse
import io
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return sorted(set(out))
    except (OSError, subprocess.SubprocessError):
        return ["unknown"]


def pil_route(srv, model, stream):
    from PIL import Image

    def perform(data, threshold):
        frame = np.array(Image.open(io.BytesIO(data)))
        return srv.perform(model, stream, frame, threshold)
    return perform


def run_once(srv, route, payloads, stream_models, thresholds, seconds, warmup):
    lat = [[] for _ in stream_models]
    phase = [0]  # 0 warm-up, 1 measuring, 2 stop
    errors = []

    def client(s):
        model = stream_models[s]
        perform = srv.detector(model, s).perform if route == "device" else pil_route(srv, model, s)
        data = payloads[model]
        k = s * 7
        try:
            while phase[0] < 2:
                t0 = time.perf_counter()
                perform(data[k % len(data)], thresholds[s])
                t1 = time.perf_counter()
                if phase[0] == 1:
                    lat[s].append((t1 - t0) * 1e3)
                k += 1
        except Exception as e:  # noqa: BLE001
            errors.append(repr(e))

    threads = [threading.Thread(target=client, args=(s,)) for s in range(len(stream_models))]
    for t in threads:
        t.start()
    time.sleep(warmup)
    stats0, cpu0, t_start = srv.lane_stats(), os.times(), time.perf_counter()
    phase[0] = 1
    time.sleep(seconds)
    phase[0] = 2
    elapsed = time.perf_counter() - t_start
    stats1, cpu1 = srv.lane_stats(), os.times()
    for t in threads:
        t.join()
    if errors:
        raise SystemExit(f"{route}: {errors[0]}")
    all_lat = np.sort(np.concatenate([np.asarray(x) for x in lat]))
    batches = sum(stats1[k][0] - stats0[k][0] for k in stats1)
    frames = sum(stats1[k][1] - stats0[k][1] for k in stats1)
    cpu = (cpu1.user - cpu0.user) + (cpu1.system - cpu0.system)
    return {"route": route, "frames_per_second": round(len(all_lat) / elapsed, 1),
            "latency_ms": {"p50": round(float(np.percentile(all_lat, 50)), 2), "p99": round(float(np.percentile(all_lat, 99)), 2)},
            "mean_batch": round(frames / max(batches, 1), 2), "host_cpu_ms_per_frame": round(1e3 * cpu / max(len(all_lat), 1), 3),
            "frames": int(len(all_lat)), "seconds": round(elapsed, 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", default="64,256")
    ap.add_argument("--seconds", type=float, default=5.0)
    ap.add_argument("--warmup", type=float, default=1.5)
    ap.add_argument("--rounds", type=int, default=2, help="pil / device alternations per setting")
    ap.add_argument("--max-batch", type=int, default=64)
    ap.add_argument("--out", help="also write the JSON lines here")
    args = ap.parse_args()
    from PIL import Image

    from fastdet_b200 import _native, modelgen
    from fastdet_b200.server import DetectServer
    gpus = _native.device_count()
    if gpus < 1:
        raise SystemExit("serve_jpeg needs a CUDA device (there is no CPU fallback)")
    specs = {"full": (modelgen.build_onnx("full", 80, 416, 2), 80), "rsu": (modelgen.build_onnx("rsu", 9, 416, 3), 9)}
    names = list(specs)
    srv = DetectServer(specs, devices=range(gpus), max_batch=args.max_batch, max_det=256)
    srv.warm(args.max_batch)
    payloads = {}
    for i, n in enumerate(names):
        payloads[n] = []
        for j in range(16):
            buf = io.BytesIO()
            Image.fromarray(modelgen.synthetic_frame(6000 + 100 * i + j, 416)).save(buf, "JPEG", quality=85)
            payloads[n].append(buf.getvalue())
    base_thr = {"full": 0.3, "rsu": 0.1}
    other = {"full": "rsu", "rsu": "full"}
    lines = []
    head = {"gpus": gpus, "gpu": gpu_identity(), "models": {n: specs[n][1] for n in names}, "max_batch": args.max_batch}
    print(json.dumps(head), flush=True)
    lines.append(head)
    for streams in [int(s) for s in args.streams.split(",")]:
        stream_models = [names[(s // gpus) % len(names)] for s in range(streams)]
        for variant in ("per_model", "mixed"):
            thresholds = []
            seen = {n: 0 for n in names}
            for m in stream_models:
                use = other[m] if variant == "mixed" and seen[m] % 2 else m
                thresholds.append(base_thr[use])
                seen[m] += 1
            for r in range(args.rounds):
                for route in ("pil", "device"):
                    res = run_once(srv, route, payloads, stream_models, thresholds, args.seconds, args.warmup)
                    res.update({"streams": streams, "thresholds": variant, "round": r})
                    print(json.dumps(res), flush=True)
                    lines.append(res)
    srv.close()
    if args.out:
        with open(args.out, "w") as fp:
            for ln in lines:
                fp.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
