"""Cost of supersampled anti-aliasing (maray_cuda_set_samples) on one GPU.

    python tools/supersample_bench.py [--samples 1,2,4] [--steps 10] [--warmup 3] [--out FILE]

For each workload (chess_4k, sdf at 1920x1080; NVRTC back end) and each s, one handle renders the whole frame with
maray_cuda_render_band into a device buffer, timed with CUDA events around every step, the L2 flushed (256 MiB memset)
between steps outside the event pairs, as bench.py does.  Reports ms per frame, Mpixel/s, Msample/s and
t(s) / (s^2 * t(1)): 1.0 means a sample costs what a pixel of the one-sample frame costs.  The card's name and power
limit are read in the same run.  Prints one JSON document (and writes it to --out)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
os.environ.setdefault("MARAY_JIT_CACHE", os.path.join(tempfile.gettempdir(), "maray_b200_supersample_bench"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", default="1,2,4")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch

    from maray_b200 import CudaRenderer, scenes

    if not torch.cuda.is_available():
        raise SystemExit("supersample_bench: no CUDA device (the render path has no CPU fallback)")
    samples = [int(v) for v in args.samples.split(",")]
    assert samples[0] == 1, "the ratio is taken against s = 1: list it first"
    workloads = [("chess_4k", scenes.chess_4k(), 3840, 2160), ("sdf", scenes.sdf(), 1920, 1080)]
    stream = torch.cuda.Stream()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    doc = {"card": card(), "backend": "nvrtc", "steps": args.steps, "warmup": args.warmup,
           "timing": "CUDA events around each render_band of the whole frame; L2 flushed between steps", "results": []}
    for name, scene, w, h in workloads:
        frame = torch.empty(w * h * 3, dtype=torch.uint8, device="cuda")
        with CudaRenderer(gpus=1) as r:
            r.load(scene)
            st = r.compile("nvrtc")
            t1 = None
            for s in samples:
                r.set_samples(s)
                for _ in range(args.warmup):
                    r.render_band(w, h, 0, h, frame.data_ptr(), stream.cuda_stream)
                    with torch.cuda.stream(stream):
                        flush.zero_()
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
                for a, b in ev:
                    a.record(stream)
                    r.render_band(w, h, 0, h, frame.data_ptr(), stream.cuda_stream)
                    b.record(stream)
                    with torch.cuda.stream(stream):
                        flush.zero_()
                stream.synchronize()
                per = [a.elapsed_time(b) for a, b in ev]
                ms = sum(per) / len(per)
                if s == 1:
                    t1 = ms
                row = {"workload": name, "width": w, "height": h, "samples": s, "passes": s * s, "ms_per_frame": ms,
                       "ms_min": min(per), "ms_max": max(per), "mpixel_per_s": w * h / ms / 1e3,
                       "msample_per_s": w * h * s * s / ms / 1e3, "ratio_to_s2_t1": ms / (s * s * t1),
                       "jit_units": st["jit_units"], "jit_registers": st["jit_registers"]}
                doc["results"].append(row)
                print(json.dumps(row), file=sys.stderr, flush=True)
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
