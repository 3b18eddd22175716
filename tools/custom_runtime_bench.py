"""What a custom runtime costs against the built-in texture runtime: the `textured` workload at 3840 x 2160, rendered
with the default texture runtime and with scenes.TEXTURE_RUNTIME_SOURCE, the same functions restated as a user's
maray_app over a packed context (maray_cuda_set_functions / maray_cuda_set_context).  Both give the same bytes.

Per runtime: cold NVRTC ms (an empty cubin cache), then kernel ms per frame from the library's device events
(stats kernel_ms[0] of render_device), the two runtimes alternated frame by frame, the 126 MB L2 overwritten before every
frame.  Prints one JSON line; needs a GPU.

    python tools/custom_runtime_bench.py [--frames 40] [--warmup 5]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()

    import numpy as np
    import torch

    from maray_b200 import CudaRenderer, scenes

    scene, textures, (w, h) = scenes.by_name("textured")
    os.environ["MARAY_JIT_CACHE"] = tempfile.mkdtemp(prefix="maray_rt_bench_")   # cold NVRTC for both

    def make(kind):
        r = CudaRenderer(device_ids=[0])
        if kind == "builtin":
            r.set_textures(textures)
        else:
            r.set_functions(scenes.TEXTURE_RUNTIME_SOURCE, 5 * len(textures))
            r.set_context(scenes.pack_textures(textures))
        r.load(scene)
        st = r.compile("nvrtc")
        return r, st

    runs = {k: make(k) for k in ("builtin", "custom")}
    frames = {}
    for k, (r, _) in runs.items():
        frames[k] = r.render(w, h)
    assert np.array_equal(frames["builtin"], frames["custom"]), "the restated runtime must give the built-in bytes"

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ms = {k: [] for k in runs}
    for i in range(args.warmup + args.frames):
        for k, (r, _) in runs.items():
            flush.fill_(i & 0xFF)
            torch.cuda.synchronize()
            r.render_device(w, h)
            if i >= args.warmup:
                ms[k].append(r.stats()["kernel_ms"][0])

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    out = {"workload": "textured", "size": [w, h], "card": card, "frames": args.frames, "l2_flushed": True}
    for k, (r, st) in runs.items():
        out[k] = {"kernel_ms_median": statistics.median(ms[k]), "kernel_ms_min": min(ms[k]), "kernel_ms_max": max(ms[k]),
                  "nvrtc_ms_cold": st["nvrtc_ms"], "registers": st["jit_registers"], "cubin_bytes": st["jit_cubin_bytes"],
                  "block": st["jit_block"]}
        r.close()
    out["custom_over_builtin"] = out["custom"]["kernel_ms_median"] / out["builtin"]["kernel_ms_median"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
