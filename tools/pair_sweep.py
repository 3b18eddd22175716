"""Pixel pairs against launch shapes: is instruction-level parallelism or more warps the lever for the guarded kernel?

    python tools/pair_sweep.py [--steps 30] [--warmup 5] [--out FILE.jsonl]

For chess_4k (3840x2160) and chess_1k (1024x1024), NVRTC back end: pixel pairs on and off (MARAY_JIT_PAIRS) at the
automatic launch shape and at 640x1, 512x2 and 1024x1 (MARAY_JIT_BLOCK / MARAY_JIT_MIN_BLOCKS).  Each configuration
renders the whole frame with maray_cuda_render_band into a device buffer, timed with CUDA events around every step, the
L2 flushed (256 MiB memset) between steps outside the event pairs.  One JSON line per configuration (also appended to
--out), the card's name and power limit read in the same run."""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
os.environ.setdefault("MARAY_JIT_CACHE", os.path.join(tempfile.gettempdir(), "maray_b200_pair_sweep"))

SHAPES = [None, (640, 1), (512, 2), (1024, 1)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch

    from maray_b200 import CudaRenderer, scenes

    if not torch.cuda.is_available():
        raise SystemExit("pair_sweep: no CUDA device (the render path has no CPU fallback)")
    dev = card()
    stream = torch.cuda.Stream()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    out = open(args.out, "a") if args.out else None
    for name in ("chess_4k", "chess_1k"):
        scene, _tex, (w, h) = scenes.by_name(name)
        frame = torch.empty(w * h * 3, dtype=torch.uint8, device="cuda")
        for pairs in (1, 0):
            for shape in SHAPES:
                env = {"MARAY_JIT_PAIRS": str(pairs)}
                if shape:
                    env.update(MARAY_JIT_BLOCK=str(shape[0]), MARAY_JIT_MIN_BLOCKS=str(shape[1]))
                saved = {k: os.environ.get(k) for k in ("MARAY_JIT_PAIRS", "MARAY_JIT_BLOCK", "MARAY_JIT_MIN_BLOCKS")}
                for k in saved:
                    os.environ.pop(k, None)
                os.environ.update(env)
                try:
                    with CudaRenderer(gpus=1) as r:
                        r.load(scene)
                        r.compile("nvrtc")
                        for _ in range(args.warmup):
                            r.render_band(w, h, 0, h, frame.data_ptr(), stream.cuda_stream)
                            with torch.cuda.stream(stream):
                                flush.zero_()
                        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                              for _ in range(args.steps)]
                        for a, b in ev:
                            a.record(stream)
                            r.render_band(w, h, 0, h, frame.data_ptr(), stream.cuda_stream)
                            b.record(stream)
                            with torch.cuda.stream(stream):
                                flush.zero_()
                        stream.synchronize()
                        st = r.stats()
                finally:
                    for k, v in saved.items():
                        if v is None:
                            os.environ.pop(k, None)
                        else:
                            os.environ[k] = v
                per = sorted(a.elapsed_time(b) for a, b in ev)
                row = {"workload": name, "pairs": pairs, "shape": "auto" if shape is None else f"{shape[0]}x{shape[1]}",
                       "block": st["jit_block"], "pixels_per_thread": st["jit_pixels_per_thread"],
                       "regs": st["jit_registers"], "ms_mean": sum(per) / len(per), "ms_median": per[len(per) // 2],
                       "ms_min": per[0], "ms_max": per[-1], "nvrtc_ms": st["nvrtc_ms"],
                       "frame_sha": hashlib.sha256(frame.cpu().numpy().tobytes()).hexdigest()[:16], "card": dev}
                print(json.dumps(row), flush=True)
                if out:
                    out.write(json.dumps(row) + "\n")
                    out.flush()


if __name__ == "__main__":
    main()
