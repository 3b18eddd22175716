"""Algorithmic FP64-pipe work of a scene (the roofline numerator), SURVEY.md section 8(d).

ops(scene) = sum over the non-constant values of the un-hoisted, hash-consed program of w(op), where
w(op) is the number of FP64-pipe SASS instructions (DADD/DMUL/DFMA/DSETP) on the fast path of that
operation, read from the committed SASS of each operation compiled exactly as the back ends compile
it (profiles/sass_ops_r01.txt; regenerate with profiles/dump_op_sass.sh):

    add, mul   1   (DADD / DMUL; --fmad=false, so never a fused pair)
    neg, abs   0   (operand modifiers / integer-pipe sign ops)
    step       1   (DSETP.GE + FSEL)
    min, max   2   (DSETP.GT|LT + DSETP.NAN, 2-4 FSEL on the integer pipe)
    recip      5   (MUFU.RCP64H on the XU pipe + 5 DFMA Newton steps)
    sqrt       8   (MUFU.RSQ64H + 3 DMUL + 5 DFMA)
    sin       18   (13 DFMA + 4 DMUL + 1 DADD: reduction by pi, nine coefficients, Estrin/Horner hybrid; round 1's quadrant version was 15)
    exp       12   (8 DFMA + 2 DADD + 2 DMUL: glibc's exp, the table load not counted; round 1's polynomial was 15)
    ln        14   (9 DFMA + 3 DADD + 2 DMUL: glibc's log, table path; I2F and the table load not counted; round 1: 28)
    tex        2   (the two `< 0.0` compares; conversions and the byte load are not FP64-pipe work)

The unit is "lane-operations": one FP64-pipe instruction executed for one pixel.  The peak it is
compared with is measured on the same GPU by an FP64 issue-rate microbenchmark
(maray_cuda_fp64_peak: independent DADD/DMUL chains, no FMA), in the same unit.

This is the ALGORITHMIC count: the work the reference's evaluation performs per pixel (src/lib.rs:623-670), priced in
this build's instructions.  The generated kernels execute less where an exact rewrite applies (boolean logic, the sign
of a sine instead of the sine, step(v + c) as a comparison: DESIGN.md 3.1), so on such scenes the algorithmic fraction
can exceed 1; `executed_counts` reads what a straight-line kernel really executes from its SASS, and bench.py reports
both.
"""
from __future__ import annotations

OP_WEIGHTS = {
    "n_add": 1, "n_mul": 1, "n_neg": 0, "n_abs": 0, "n_step": 1, "n_min": 2, "n_max": 2,
    "n_recip": 5, "n_sqrt": 8, "n_sin": 18, "n_exp": 12, "n_ln": 14, "n_tex": 2,
}


def fp64_ops_per_pixel(stats: dict) -> int:
    """stats: the dict form of maray_cuda_stats after compile."""
    return sum(w * int(stats[k]) for k, w in OP_WEIGHTS.items())


def executed_counts(cubin: bytes, kernel: str = "maray_jit"):
    """FP64-pipe and total SASS instructions of `kernel` in a cubin, via `cuobjdump -sass` (None if the tool is
    missing).  For a straight-line kernel (one unit, no batched helper loops) this is what one pixel executes, the
    never-taken out-of-range blocks aside (a handful of integer instructions per sine).  None as well when the kernel
    has guarded regions (a warp vote, VOTE, in its SASS; codegen.cpp find_guard_regions): a warp runs a region's body
    only when its guard is true on some lane, so what a pixel executes depends on the frame and no longer on the code
    alone, and the static count would overstate it."""
    import os
    import re
    import shutil
    import subprocess
    import tempfile

    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        return None
    with tempfile.NamedTemporaryFile(suffix=".cubin") as f:
        f.write(cubin)
        f.flush()
        try:
            text = subprocess.run([tool, "-sass", "-fun", kernel, f.name], capture_output=True, text=True, timeout=120).stdout
        except Exception:
            return None
    fp64 = total = 0
    for m in re.finditer(r"^\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", text, flags=re.M):
        op = m.group(1)
        if op == "NOP":
            continue
        if op == "VOTE":
            return None
        total += 1
        fp64 += op in ("DFMA", "DMUL", "DADD", "DSETP")
        if op == "EXIT" and total > 64:      # end of the kernel's own path: out-of-line device functions (libdevice
            break                            # fall-backs, the checked copy of a speculated program) follow it
    return {"fp64": fp64, "all": total} if total else None
