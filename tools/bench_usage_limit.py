"""Cost of the usage limit (mosaic_set_usage_limit) on BASELINE configs 4, 5 and 3 at full size.

For each config one handle holds the inputs; the runs alternate the limits of that config (config 4: 0 / 1 / 8, config 5: 0 / 1,
config 3: 0 / 7 -- 13,823 cells over 2,000 images make 7 its smallest feasible limit) round after round, and every time is the median
of the rounds. Then one more run per limit keeps D, and the host replays the capped rule with the kernel's prefix scan on it: the grid
must equal the timed runs' grid, and the replay counts the cells whose sorted prefix ran out (the fallback to the full row).

Prints one JSON object: per config and limit the generate wall time, diff_ms, select_ms, K_s per step, the executed share of the
difference work (evaluated_pixel_diffs / pixel_diffs), the fallback count, and the GPU name and power limit read in the same process.

    python tools/bench_usage_limit.py [--rounds 3] [--configs cfg4,cfg5,cfg3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

LIMITS = {"cfg4": (0, 1, 8), "cfg5": (0, 1), "cfg3": (0, 7)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def step_bounds(cells, N, rr, ra, M):
    """K_s and the (prefix length, candidate row length) the engine uses per step (generator.cu::plan_step)"""
    from tests.helpers.usage_limit import PREFIX_MAX, exhausted_bound, k_bound
    out, before = [], 0
    for n in cells:
        K = k_bound(1, N, rr, exhausted_bound(before, n, M))
        via_topk = K * 4 <= N  # capped runs take top-K lists when they are at most a quarter of the row
        out.append((K, min(K, PREFIX_MAX), K if via_topk else N))
        before += n
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--configs", default="cfg4,cfg5,cfg3")
    ap.add_argument("--out")
    args = ap.parse_args()
    import bench
    from mosaicmagnifique_b200 import CellGroup, PhotomosaicGenerator
    from tests.helpers.usage_limit import capped_rule

    result = {"gpu": gpu_info(), "rounds": args.rounds, "configs": {}}
    for name in args.configs.split(","):
        cfg = bench.WORKLOADS[name]
        main_img, lib = bench.make_inputs(cfg)
        N = len(lib)
        gen = PhotomosaicGenerator(0)
        gen.setMainImage(main_img)
        gen.setLibrary(lib)
        gen.setColourDifference(cfg["diff"])
        cg = CellGroup()
        cg.setCellShape(bench.make_shape(cfg))
        cg.setDetail(cfg["detail"])
        cg.setSizeSteps(cfg.get("steps", 0))
        gen.setCellGroup(cg)
        state = gen.computeGridState()
        cells = [int((s >= 0).sum()) for s in state]
        gen.setRepeat(cfg["rr"], cfg["ra"])
        runs = {M: [] for M in LIMITS[name]}
        grids = {}
        for rnd in range(args.rounds + 1):  # round 0 warms every shape up and is not reported
            for M in runs:
                gen.setUsageLimit(M)
                t0 = time.perf_counter()
                assert gen.generateBestFits()
                wall = (time.perf_counter() - t0) * 1e3
                grids[M] = [g.copy() for g in gen.getBestFits()]
                if rnd:
                    runs[M].append(dict(gen.getTimings(), wall_ms=wall))
        per = {}
        for M, rs in runs.items():
            med = lambda k: float(np.median([r[k] for r in rs]))
            entry = {"generate_ms": med("wall_ms"), "preprocess_ms": med("preprocess_ms"), "diff_ms": med("diff_ms"),
                     "select_ms": med("select_ms"), "evaluated_share": med("evaluated_pixel_diffs") / med("pixel_diffs")}
            if M:
                bounds = step_bounds(cells, N, cfg["rr"], cfg["ra"], M)
                gen.setUsageLimit(M)
                gen.setKeepDifferences(True)
                assert gen.generateBestFits()
                Ds = [gen.getDifferences(s) for s in range(len(state))]
                gen.setKeepDifferences(False)
                replay, fallbacks = capped_rule(Ds, state, cfg["rr"], cfg["ra"], N, M, scan=([b[1:] for b in bounds], False))
                assert all(np.array_equal(a, b) for a, b in zip(replay, grids[M])), "replayed grid differs"
                used = np.bincount(np.concatenate([g[g >= 0] for g in grids[M]]), minlength=N)
                entry.update({"K_per_step": [b[0] for b in bounds], "prefix_per_step": [b[1] for b in bounds],
                              "candidate_row_per_step": [b[2] for b in bounds], "fallback_cells": int(fallbacks),
                              "max_uses_observed": int(used.max()), "images_used": int((used > 0).sum())})
            per[str(M)] = entry
        gen.close()
        result["configs"][name] = {"desc": cfg["desc"], "cells_per_step": cells, "images": N, "limits": per}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
