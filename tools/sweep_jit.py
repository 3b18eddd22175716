"""Sweep NVRTC back-end knobs on one workload and print kernel time per configuration (GPU box).
usage: sweep_jit.py WORKLOAD  "block,min_blocks;block,min_blocks;..."  "bank,bank"  [seg,seg]"""
import itertools, json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from maray_b200 import CudaRenderer, scenes
from maray_b200.roofline import fp64_ops_per_pixel

workload = sys.argv[1] if len(sys.argv) > 1 else "chess_4k"
shapes = [tuple(x.split(",")) for x in (sys.argv[2] if len(sys.argv) > 2 else "256,2;256,3;128,4;128,5;128,6").split(";")]
banks = (sys.argv[3] if len(sys.argv) > 3 else "1,0").split(",")
segs = (sys.argv[4] if len(sys.argv) > 4 else "32768").split(",")
scene, tex, (w, h) = scenes.by_name(workload)
peak = None
for (block, minb), bank, seg in itertools.product(shapes, banks, segs):
    os.environ.update({"MARAY_JIT_BLOCK": block, "MARAY_JIT_MIN_BLOCKS": minb, "MARAY_JIT_CONST_BANK": bank,
                       "MARAY_JIT_SEGMENT_VALUES": seg})
    with CudaRenderer(gpus=1) as r:
        if peak is None:
            peak = r.fp64_peak(0)[0]
        r.set_textures(tex); r.load(scene)
        st = r.compile("nvrtc")
        ops = fp64_ops_per_pixel(st)
        best = 1e9
        for i in range(4):
            r.render_device(w, h)
            best = min(best, r.stats()["kernel_ms"][0])
        print(json.dumps({"block": block, "minb": minb, "bank": bank, "seg": seg, "regs": st["jit_registers"],
                          "nvrtc_ms": round(st["nvrtc_ms"]), "kernel_ms": round(best, 3), "mpix_s": round(w * h / best / 1e3, 1),
                          "frac": round(w * h * ops / (best * 1e-3) / peak, 3)}), flush=True)
