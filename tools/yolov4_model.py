#!/usr/bin/env python
"""YOLOv4-416 on one GPU: forward time and its share of the bf16 burst peak, fd_detect frames/s, each Mish layer next to the
same layer of the LeakyReLU twin graph, and the SPP launch.

    python tools/yolov4_model.py [--reps 20] [--json out.json] [--pools-only]

Forward time is fd_time_forward (device events around the conv stack, frames already on the device); the share of burst is
the conv FLOPs over that time against the 1670.5 TFLOP/s burst bf16 rate measured on a B200 (DESIGN.md §3).  fd_detect is the
synchronous call from pinned host frames, timed with a host clock over `--reps` calls after a warm-up.  Per-layer times come
from fd_time_layers (each layer's own launch, timed alone).  The twin (ExportOptions(mish_as_leaky=True)) is the same graph
with LeakyReLU(0.1) in place of every Mish; the fused stem and block take its first layers, so the Mish layers 0, 1, 4 and 5
have no twin of their own.  The SPP line is the group's one launch; --pools-only prints the three pool layers of the twin
alone, which is how a build without the SPP kernel (one maxpool_kernel launch per pool) is timed."""
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

BURST = 1670.5e12  # bf16 FLOP/s, measured burst peak of one B200 (DESIGN.md §3)


def gpu():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          stdout=subprocess.PIPE, text=True, check=True).stdout.strip()


def measure(n, reps, twin=False, size=416):
    opts = modelgen.ExportOptions(mish_as_leaky=True) if twin else None
    m = _native.Model(modelgen.build_onnx("v4", 80, size, seed=1, opts=opts), 80, (size, size), device=0)
    host = torch.from_numpy(np.stack([modelgen.synthetic_frame(100 + i % 4, size) for i in range(n)])).pin_memory().numpy()
    m.preprocess(host, n, (size, size))
    m.forward(n)
    fwd_ms = float(m.time_forward(n, reps))
    layer_ms = [float(v) for v in m.time_layers(n, reps)]
    info = m.exec_info(n)
    L = m.layers()
    for _ in range(3):
        m.detect(host, 0.1)
    t0 = time.perf_counter()
    for _ in range(reps):
        m.detect(host, 0.1)
    det_s = (time.perf_counter() - t0) / reps
    row = dict(batch=n, twin=twin, forward_ms=fwd_ms, burst_share=m.info.conv_flops_per_frame * n / (fwd_ms * 1e-3) / BURST,
               detect_fps=n / det_s, layers=[dict(name=l["name"], kind=l["kind"], act=l["act"], kernel=e["kernel_name"], split_k=e["split_k"],
                                                 us=t * 1e3, h=l["h"], cin=l["cin"], c=l["c"], k=l["ksize"], s=l["stride"])
                                            for l, e, t in zip(L, info, layer_ms)])
    m.close()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--json", default="")
    ap.add_argument("--pools-only", action="store_true")
    a = ap.parse_args()
    print("GPU 0 (name, power limit):", gpu())
    out = []
    for n in (1, 64):
        if a.pools_only:
            t = measure(n, a.reps, twin=True)
            pools = [l for l in t["layers"] if l["kind"] == 2]
            print(f"batch {n}: pool launches " + ", ".join(f"{l['name']} {l['kernel']} {l['us']:.1f} us" for l in pools)
                  + f"; sum {sum(l['us'] for l in pools):.1f} us")
            out.append(t)
            continue
        mish, leaky = measure(n, a.reps), measure(n, a.reps, twin=True)
        out += [mish, leaky]
        for r in (mish, leaky):
            print(f"batch {n:2d} {'leaky twin' if r['twin'] else 'YOLOv4    '}: forward {r['forward_ms']:.3f} ms "
                  f"({r['burst_share']:.1%} of burst), fd_detect {r['detect_fps']:.0f} frames/s")
        print(f"  {'layer':<8} {'map':>4} {'cin':>5} {'cout':>5} k s  {'Mish form':<14} {'Mish us':>8} {'leaky us':>8} {'ratio':>6}")
        tot_m = tot_l = 0.0
        for lm, ll in zip(mish["layers"], leaky["layers"]):
            if lm["act"] != 2:
                continue
            twin_ok = ll["kernel"] not in ("fused_next", "stem", "block")
            form = lm["kernel"] + (" s2" if lm["s"] == 2 and lm["kernel"] == "halo" else "") + (f" sk{lm['split_k']}" if lm["split_k"] > 1 else "")
            if twin_ok:
                tot_m += lm["us"]
                tot_l += ll["us"]
            print(f"  {lm['name']:<8} {lm['h']:4d} {lm['cin']:5d} {lm['c']:5d} {lm['k']} {lm['s']}  {form:<14} {lm['us']:8.1f} "
                  + (f"{ll['us']:8.1f} {lm['us'] / ll['us']:6.2f}" if twin_ok else f"{'(' + ll['kernel'] + ')':>15}"))
        print(f"  Mish layers with a twin: {tot_m:.1f} us against {tot_l:.1f} us leaky (+{tot_m - tot_l:.1f} us)")
        spp = [l for l in mish["layers"] if l["kernel"] == "spp"]
        print(f"  SPP: one launch {spp[0]['us']:.1f} us" if spp else "  SPP: not grouped")
    if a.json:
        with open(a.json, "w") as fp:
            json.dump(dict(gpu=gpu(), rows=out), fp, indent=1)


if __name__ == "__main__":
    main()
