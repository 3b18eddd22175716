"""Cost of PNG output per workload: maray_cuda_render_png against rendering into a pageable image and encoding on the
host the way write_png_rgb8 does (filter None, zlib level 6).  One JSON line per workload, plus the card's name and
power limit, to stdout or --out.

    python tools/png_bench.py [--workloads chess_4k,chess_1k,sdf,textured,deep] [--reps 5] [--out file.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from maray_b200 import CudaRenderer, scenes  # noqa: E402


def host_png(img):
    """write_png_rgb8's bytes: scanlines with filter None, zlib level 6, one IDAT."""
    h, w = img.shape[:2]
    raw = np.concatenate([np.zeros((h, 1), np.uint8), img.reshape(h, 3 * w)], axis=1).tobytes()
    return 57 + len(zlib.compress(raw, 6))


def idat_level6(png):
    """Level 6 over the GPU file's own (adaptively filtered) scanlines."""
    pos, z = 8, b""
    while pos < len(png):
        n = int.from_bytes(png[pos:pos + 4], "big")
        if png[pos + 4:pos + 8] == b"IDAT":
            z += png[pos + 8:pos + 8 + n]
        pos += 12 + n
    return 57 + len(zlib.compress(zlib.decompress(z), 6))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="chess_4k,chess_1k,sdf,textured,deep")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = open(a.out, "w") if a.out else sys.stdout
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps({"card": card[0] if card else "unknown"}), file=out, flush=True)
    for name in a.workloads.split(","):
        scene, tex, (w, h) = scenes.by_name(name)
        reps = 1 if name == "deep" else a.reps
        with CudaRenderer(gpus=1) as r:
            r.set_textures(tex)
            r.load(scene)
            r.compile("nvrtc")
            png, _, ps = r.render_png(w, h)          # warm-up: scratch, pinned buffer
            img = np.zeros((h, w, 3), np.uint8)
            r.render_into(img)
            new_t, enc, old_t = [], [], []
            for _ in range(reps):
                t0 = time.perf_counter()
                png, _, ps = r.render_png(w, h)
                new_t.append(time.perf_counter() - t0)
                enc.append(ps["encode_ms"])
                t0 = time.perf_counter()
                r.render_into(img)
                old_bytes = host_png(img)
                old_t.append(time.perf_counter() - t0)
        rec = {"workload": name, "w": w, "h": h, "segments": ps["segments"], "stored_segments": ps["stored_segments"],
               "scanline_bytes": ps["scanline_bytes"], "encode_ms": min(enc),
               "encode_GBps": ps["scanline_bytes"] / (min(enc) * 1e6), "d2h_ms": ps["d2h_ms"],
               "render_png_wall_ms": 1e3 * min(new_t), "render_then_host_png_wall_ms": 1e3 * min(old_t),
               "png_bytes": ps["png_bytes"], "host_png_bytes": old_bytes, "level6_same_filters_bytes": idat_level6(png)}
        print(json.dumps(rec), file=out, flush=True)


if __name__ == "__main__":
    main()
