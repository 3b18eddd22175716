"""Predicted SASS instructions per pixel of a straight-line kernel with guarded regions, without a GPU.

    python tools/guard_regions_predict.py [--workload chess_4k] [--row-step 16]

1. The scene is compiled through NVRTC (no device needed) and its SASS read with `cuobjdump -sass` (CUDA toolkit): each `VOTE` is
   followed by the conditional branch that skips the region's body; the instructions between that branch and its
   target are the body's static count (nested bodies included in their outer one).
2. The generated text is built for the host with every region evaluated at every pixel, and each vote records its
   guard.  Over whole 32-pixel warps of a sample of rows (a warp runs a body when the guard is true on one of its
   lanes and, for a nested region, its outer body runs) this gives how often each body runs.
3. Executed per pixel = static count of the kernel's own path - the bodies a warp skips.

Regions in the text and in the SASS are matched in order; the script checks that their nesting agrees.  Prints one
JSON line."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ.setdefault("MARAY_JIT_CACHE", "off")

VOTE = "if (mr_warp_any("


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="chess_4k")
    ap.add_argument("--row-step", type=int, default=16, help="sample every N-th row of the frame")
    args = ap.parse_args()
    from helpers import HOST_SHIM
    from maray_b200 import CudaRenderer, scenes

    scene, textures, (w, h) = scenes.by_name(args.workload)
    assert w % 32 == 0, "rows must hold whole warps"
    with CudaRenderer(gpus=0) as r:
        r.set_textures(list(textures))
        r.load(scene)
        r.compile("nvrtc")
        src, cubin = r.source(), r.cubin(0)
    tmp = tempfile.mkdtemp(prefix="maray_guard_predict_")

    # regions of the text and their nesting
    parts = src.split(VOTE)
    n_reg = len(parts) - 1
    parent, stack = [], []
    for line in src[src.index('extern "C" __global__'):].splitlines():
        if line.startswith("  " + VOTE):
            parent.append(stack[-1] if stack else -1)
            stack.append(len(parent) - 1)
        elif line == "  }":
            stack.pop()
    assert len(parent) == n_reg

    # regions of the SASS: VOTE, then the predicated branch over the body
    with open(os.path.join(tmp, "k.cubin"), "wb") as f:
        f.write(cubin)
    sass = subprocess.run(["cuobjdump", "-sass", os.path.join(tmp, "k.cubin")], capture_output=True, text=True, check=True).stdout
    ins = []
    for m in re.finditer(r"^\s+/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z0-9_.]+)([^;]*);", sass, flags=re.M):
        ins.append((int(m.group(1), 16), bool(m.group(2)), m.group(3), m.group(4)))
        if m.group(3) == "EXIT" and len(ins) > 64:
            break
    at = {a: i for i, (a, *_rest) in enumerate(ins)}
    spans = []
    for i, (_a, _p, op, _r) in enumerate(ins):
        if op.startswith("VOTE"):
            j = next(j for j in range(i + 1, len(ins)) if ins[j][2].startswith("BRA") and ins[j][1])
            spans.append((j, at[int(re.search(r"0x([0-9a-f]+)", ins[j][3]).group(1), 16)]))
    assert len(spans) == n_reg, (len(spans), n_reg)
    sass_parent, stack = [], []
    for k, (j, t) in enumerate(spans):
        while stack and not (spans[stack[-1]][0] < j < spans[stack[-1]][1]):
            stack.pop()
        sass_parent.append(stack[-1] if stack else -1)
        stack.append(k)
    assert sass_parent == parent, "regions of the text and of the SASS do not nest alike"
    count = lambda lo, hi: sum(1 for x in ins[lo:hi] if x[2] != "NOP")
    total = count(0, len(ins))
    body = np.array([count(j + 1, t) for j, t in spans])
    own = body.copy()                                   # a body's instructions outside its nested bodies
    for k, p in enumerate(parent):
        if p >= 0:
            own[p] -= body[k]

    # guards per pixel from the host build, every body evaluated
    text = parts[0] + "".join(f"if (mr_rec({i}, " + p for i, p in enumerate(parts[1:]))
    text = text.replace('extern "C" __global__', "static")
    cut = text.index("static void __launch_bounds__")
    text = (text[:cut] + f"static unsigned char g_guard[{n_reg}];\n"
            "static inline bool mr_rec(int k, bool b) { g_guard[k] = b; return true; }\n" + text[cut:])
    driver = r"""
extern "C" void guards_of_row(unsigned int W, unsigned int y, unsigned char* rec) {
    unsigned char out[3];
    MrParams p; std::memset(&p, 0, sizeof p);
    p.out = out; p.n = 1; p.W = W;
    blockDim.x = 1; blockIdx.x = 0; threadIdx.x = 0;
    for (unsigned int x = 0; x < W; x++) {
        p.p0 = y * W + x;
        maray_jit(p);
        std::memcpy(rec + (size_t)x * NREG, g_guard, NREG);
    }
}
""".replace("NREG", str(n_reg))
    with open(os.path.join(tmp, "k.cpp"), "w") as f:
        f.write("#define MR_HOST_GUARDS_ALWAYS 1\n" + HOST_SHIM + text + driver)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-w",
                           "-o", os.path.join(tmp, "k.so"), os.path.join(tmp, "k.cpp")])
    lib = ctypes.CDLL(os.path.join(tmp, "k.so"))
    runs = []
    for y in range(0, h, args.row_step):
        rec = np.zeros((w, n_reg), np.uint8)
        lib.guards_of_row(w, y, rec.ctypes.data)
        vote = rec.reshape(w // 32, 32, n_reg).any(axis=1)
        run = np.zeros_like(vote)
        for k, p in enumerate(parent):                   # outer regions come first
            run[:, k] = vote[:, k] & (run[:, p] if p >= 0 else True)
        runs.append(run)
    run = np.concatenate(runs)
    executed = total - (own[None, :] * ~run).sum(axis=1)
    top = body[[p < 0 for p in parent]]
    print(json.dumps({
        "workload": args.workload, "regions": n_reg, "nested": int(sum(p >= 0 for p in parent)),
        "static_instructions": total, "static_in_bodies": int(own.sum()),
        "top_body_instructions_min_median_max": [int(top.min()), float(np.median(top)), int(top.max())],
        "warps_sampled": int(run.shape[0]), "bodies_run_per_warp": float(run.sum(axis=1).mean()),
        "warps_running_0_1_2plus_top_bodies": [float(v) for v in np.bincount(np.minimum(run[:, [p < 0 for p in parent]].sum(axis=1), 2), minlength=3) / run.shape[0]],
        "predicted_executed_per_pixel": float(executed.mean()), "fraction_of_static": float(executed.mean() / total),
        "worst_warp_fraction": float(executed.max() / total)}))


if __name__ == "__main__":
    main()
