#!/usr/bin/env python3
"""Instruction counts of the difference kernels' inner loops, taken from the SASS of the built library.

    python tools/sass_counts.py            # writes profiles/r2_sass_<kernel>.txt (loop listing) and profiles/r2_sass_counts.json

For each hot kernel the consumer loop is the largest INNERMOST backward-branch loop of the function (`BRA[.U] ... <lower address>`,
mbarrier spin loops ignored). Its body
is listed and classified per pipe; the counts are per THREAD per loop iteration and are divided by the pixel-differences one lane
produces per iteration (stated per kernel below) to give the executed work per pixel-difference that bench.py's roofline uses:

    packed FP32 (FFMA2 / FMUL2 / FADD2)  : 2 FP32 lane-ops each, FMA-heavy pipe, 2 issue cycles
    scalar FP32 (FFMA / FMUL / FADD ...) : 1 lane-op
    MUFU.*                               : XU pipe (16 lanes / clk / SM)
bench.py reads profiles/r2_sass_counts.json (committed; regenerate after every kernel change) and, where cuobjdump is available,
re-derives the counts from the library it actually loaded and reports whether they agree (the build is not byte-reproducible, so
counts are compared, not file hashes).
"""
import hashlib
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "mosaicmagnifique_b200", "libmosaic_b200.so")

# kernel name pattern -> (short name, pixel-differences per lane per loop iteration, how that is derived)
KERNELS = {
    # the CIEDE2000 launches that write D (every penalised / top-K step) run diff_rows_kernel; its consumer loop is the same code as
    # diff_sum_kernel's (consume_ring), which now only serves the fused-argmin launch
    r"diff_rows_kernel": ("diff_sum", 8, "one pixel of the lane's cell x the 8 library images of the tile (4 packed pairs), diff_kernels.cu diff_rows_kernel"),
    r"diff_euclid_kernel": ("diff_euclid", None, "4 cells x 4 images per pixel, x the loop's pixel unroll (derived from the MUFU.SQRT count: 1 per pair)"),
}
PACKED = ("FFMA2", "FMUL2", "FADD2")
SCALAR_FP32 = ("FFMA", "FMUL", "FADD")  # FMA pipe; FSEL / FSETP / FMNMX issue on the ALU pipe and are counted with alu_other


def functions(sass):
    cur, out = None, {}
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
        elif cur and re.match(r"\s+/\*[0-9a-f]{4,}\*/", line):
            m2 = re.match(r"\s+/\*([0-9a-f]+)\*/\s+(.*?);", line)
            if m2:
                out[cur].append((int(m2.group(1), 16), m2.group(2).strip()))
    return out


def hot_loop(instrs):
    """The innermost substantial loop: among the backward-branch loops that enclose no other loop of >= 20 instructions (the
    two-instruction mbarrier try_wait spins do not count as loops) the one with the most MUFU instructions -- the consumer loop; the
    producer's unrolled TMA loop has none."""
    loops = []
    for addr, text in instrs:
        m = re.search(r"\bBRA(?:\.\S+)?\s+(?:!?U?P\d+,\s*)?(0x[0-9a-f]+)", text)
        if m:
            tgt = int(m.group(1), 16)
            if tgt < addr:
                loops.append((tgt, addr))
    big = [l for l in loops if (l[1] - l[0]) // 16 + 1 >= 20]
    inner = [l for l in big if not any(o != l and l[0] <= o[0] and o[1] <= l[1] for o in big)]
    mufu = lambda l: sum(1 for a, t in instrs if l[0] <= a <= l[1] and "MUFU" in t)
    return max(inner, key=lambda l: (mufu(l), l[1] - l[0]))


def classify(body):
    c = {"packed_fp32": 0, "scalar_fp32": 0, "mufu": 0, "lds": 0, "alu_other": 0, "control": 0, "total": 0}
    ops = {}
    for _, text in body:
        t = re.sub(r"^@!?U?P\d+\s+", "", text)
        op = t.split()[0]
        base = op.split(".")[0]
        ops[base] = ops.get(base, 0) + 1
        c["total"] += 1
        if base in PACKED:
            c["packed_fp32"] += 1
        elif base in SCALAR_FP32:
            c["scalar_fp32"] += 1
        elif base == "MUFU":
            c["mufu"] += 1
        elif base in ("LDS", "LDSM"):
            c["lds"] += 1
        elif base in ("BRA", "WARPSYNC", "NOP", "YIELD", "BSSY", "BSYNC", "EXIT"):
            c["control"] += 1
        else:
            c["alu_other"] += 1
    return c, ops


def analyse(lib=LIB, write_listings=False):
    """Counts of the hot loops of `lib`. The build is not byte-reproducible (nvcc embeds unique ids), so consumers compare COUNTS,
    not file hashes: bench.py re-runs this on the library it loaded and checks it against the committed JSON."""
    sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs = functions(sass)
    sha = hashlib.sha256(open(lib, "rb").read()).hexdigest()
    result = {"library": os.path.relpath(lib, ROOT), "library_sha256": sha, "arch": "sm_100a" if "sm_100a" in sass else "?", "kernels": {}}
    whole = {}
    for instrs in funcs.values():
        for _, t in instrs:
            base = re.sub(r"^@!?U?P\d+\s+", "", t).split()[0].split(".")[0]
            if base in ("UBLKCP", "UTMALDG", "SYNCS", "FFMA2", "FMUL2", "FADD2", "MUFU"):
                whole[base] = whole.get(base, 0) + 1
    result["whole_library_mnemonics"] = whole
    for pat, (short, per_iter, how) in KERNELS.items():
        match = [n for n in funcs if re.search(pat, n)]
        if not match:
            print("kernel %s not found" % pat, file=sys.stderr)
            continue
        fn = match[0]
        instrs = funcs[fn]
        lo, hi = hot_loop(instrs)
        body = [(a, t) for a, t in instrs if lo <= a <= hi]
        c, ops = classify(body)
        if per_iter is None:
            per_iter = c["mufu"]  # Euclidean: exactly one MUFU.SQRT per pixel-difference
        lane_ops = 2 * c["packed_fp32"] + c["scalar_fp32"]
        k = {"function": fn, "loop": [hex(lo), hex(hi)], "pixel_diffs_per_lane_per_iteration": per_iter, "how": how, "counts": c,
             "opcodes": dict(sorted(ops.items(), key=lambda kv: -kv[1])),
             "per_pixel_diff": {"fp32_lane_ops": lane_ops / per_iter, "mufu": c["mufu"] / per_iter,
                                "packed_fp32_instr": c["packed_fp32"] / per_iter, "scalar_fp32_instr": c["scalar_fp32"] / per_iter,
                                "other_instr": (c["alu_other"] + c["lds"] + c["control"]) / per_iter,
                                # one warp instruction per clock per sub-partition; a packed FP32 instruction holds the FP32 pipe for two
                                "dispatch_or_pipe_cycles": (2 * c["packed_fp32"] + c["total"] - c["packed_fp32"]) / per_iter},
             "tma_mbarrier_in_function": {op: sum(1 for _, t in instrs if re.sub(r"^@!?U?P\d+\s+", "", t).split()[0].split(".")[0] == op)
                                          for op in ("UBLKCP", "SYNCS")}}
        result["kernels"][short] = k
        if not write_listings:
            continue
        path = os.path.join(ROOT, "profiles", "r2_sass_%s.txt" % short)
        with open(path, "w") as f:
            f.write("# cuobjdump -sass %s  -- function %s\n" % (result["library"], fn))
            f.write("# library sha256 %s\n" % sha)
            f.write("# inner (consumer) loop %s..%s: %d instructions per iteration, %s pixel-differences per lane per iteration (%s)\n"
                    % (hex(lo), hex(hi), c["total"], per_iter, how))
            f.write("# counts per iteration: %s\n" % json.dumps(c))
            f.write("# per pixel-difference: %s\n" % json.dumps(k["per_pixel_diff"]))
            f.write("# TMA / mbarrier instructions in the whole function: %s\n" % json.dumps(k["tma_mbarrier_in_function"]))
            f.write("# opcode histogram of the loop: %s\n#\n" % json.dumps(k["opcodes"]))
            for a, t in instrs:
                mark = "L " if lo <= a <= hi else "  "
                f.write("%s/*%04x*/ %s ;\n" % (mark, a, t))
        print("%s: loop %s..%s  %s  per pixel-diff %s" % (short, hex(lo), hex(hi), c, k["per_pixel_diff"]))
    return result


def main():
    result = analyse(LIB, write_listings=True)
    with open(os.path.join(ROOT, "profiles", "r2_sass_counts.json"), "w") as f:
        json.dump(result, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
