#!/usr/bin/env python
"""YOLOv3-tiny and YOLOv4-tiny side by side on one GPU: forward time, fd_detect frames/s from pinned host frames, and the
first layer's time next to its HBM bound.

    python tools/tiny_models.py [--reps 20] [--json out.json]

Forward time is fd_time_forward (device events around the conv stack, frames already on the device).  fd_detect is the
synchronous call a server makes: pinned host frames in (copy overlapped with the first layers), detection records out,
timed with a host clock over `--reps` calls after a warm-up.  The first layer's time is its own launch from fd_time_layers;
its HBM bound is the u8 frames it reads plus the bf16 tensor it writes, at the data sheet's 7.7 TB/s."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fastdet_b200 import _native, modelgen  # noqa: E402

HBM = 7.7e12  # bytes/s, HGX B200 data sheet, one GPU


def gpu():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         stdout=subprocess.PIPE, text=True, check=True).stdout.strip()
    return out


def measure(arch, n, reps, size=416):
    data = modelgen.build_onnx(arch, 80, size, seed=1)
    m = _native.Model(data, 80, (size, size), device=0)
    frames = torch.from_numpy(np.stack([modelgen.synthetic_frame(100 + i % 4, size) for i in range(n)])).pin_memory()
    host = frames.numpy()
    m.preprocess(host, n, (size, size))
    m.forward(n)
    fwd_ms = m.time_forward(n, reps)
    layer_ms = m.time_layers(n, reps)
    L = m.layers()
    for _ in range(3):
        m.detect(host, 0.1)
    t0 = time.perf_counter()
    for _ in range(reps):
        m.detect(host, 0.1)
    det_s = (time.perf_counter() - t0) / reps
    l0 = L[0]
    bytes0 = n * size * size * 3 + n * l0["h"] * l0["w"] * l0["c"] * 2
    row = dict(arch=arch, batch=n, forward_ms=float(fwd_ms), detect_fps=n / det_s, layer0_us=float(layer_ms[0]) * 1e3,
               layer0_stride=l0["stride"], layer0_hbm_bound_us=bytes0 / HBM * 1e6, kernel0=m.exec_info(n)[0]["kernel_name"],
               launches=m.info.n_layers)
    m.close()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--json", default="")
    a = ap.parse_args()
    print("GPU 0 (name, power limit):", gpu())
    rows = []
    print(f"{'arch':<6} {'batch':>5} {'launches':>8} {'forward ms':>10} {'detect fr/s':>11} {'layer0':>12} {'us':>8} {'HBM bound us':>12} {'share':>6}")
    for arch in ("tiny", "tiny4"):
        for n in (1, 64):
            r = measure(arch, n, a.reps)
            rows.append(r)
            print(f"{arch:<6} {n:5d} {r['launches']:8d} {r['forward_ms']:10.3f} {r['detect_fps']:11.0f} "
                  f"{r['kernel0'] + (' s2' if r['layer0_stride'] == 2 else ' s1+pool'):>12} {r['layer0_us']:8.1f} "
                  f"{r['layer0_hbm_bound_us']:12.1f} {r['layer0_hbm_bound_us'] / r['layer0_us']:6.1%}")
    if a.json:
        with open(a.json, "w") as fp:
            json.dump(dict(gpu=gpu(), rows=rows), fp, indent=1)


if __name__ == "__main__":
    main()
