"""Cost of mirrored library tiles (mosaic_set_tile_flips) on BASELINE configs 4 and 5 at full size.

For each config one handle holds the inputs; the runs alternate flips 0 / 1 / 3 (horizontal, horizontal + vertical) round after
round, and every number is the median of the rounds. Because the flips change between consecutive runs, every flips > 0 run
rebuilds the oriented library, so `preprocess_ms` includes that cost (its worst case: a run after a change of library or flips).

Prints one JSON object: per config and flips the generate wall time, the phase times, the slot count O * N and
evaluated_pixel_diffs / pixel_diffs (the share of the difference work that exact pruning left), with the GPU name and power limit
read in the same process.

    python tools/bench_tile_flips.py [--rounds 3] [--out FILE]
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


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--configs", default="cfg4,cfg5")
    ap.add_argument("--out")
    args = ap.parse_args()
    import bench
    from mosaicmagnifique_b200 import CellGroup, PhotomosaicGenerator

    result = {"gpu": gpu_info(), "rounds": args.rounds, "configs": {}}
    for name in args.configs.split(","):
        cfg = bench.WORKLOADS[name]
        main_img, lib = bench.make_inputs(cfg)
        gen = PhotomosaicGenerator(0)
        gen.setMainImage(main_img)
        gen.setLibrary(lib)
        gen.setColourDifference(cfg["diff"])
        cg = CellGroup()
        cg.setCellShape(bench.make_shape(cfg))
        cg.setDetail(cfg["detail"])
        cg.setSizeSteps(cfg.get("steps", 0))
        gen.setCellGroup(cg)
        gen.computeGridState()
        gen.setRepeat(cfg["rr"], cfg["ra"])
        runs = {f: [] for f in (0, 1, 3)}
        for rnd in range(args.rounds + 1):  # round 0 warms every shape up and is not reported
            for f in runs:
                gen.setTileFlips(bool(f & 1), bool(f & 2))
                t0 = time.perf_counter()
                assert gen.generateBestFits()
                wall = (time.perf_counter() - t0) * 1e3
                if rnd:
                    runs[f].append(dict(gen.getTimings(), wall_ms=wall))
        gen.close()
        per = {}
        for f, rs in runs.items():
            med = lambda k: float(np.median([r[k] for r in rs]))
            per[str(f)] = {"slots": len(lib) << bin(f).count("1"), "generate_ms": med("wall_ms"), "preprocess_ms": med("preprocess_ms"),
                           "diff_ms": med("diff_ms"), "select_ms": med("select_ms"),
                           "evaluated_share": med("evaluated_pixel_diffs") / med("pixel_diffs"), "pixel_diffs": med("pixel_diffs")}
        base = per["0"]["diff_ms"]
        for f in per:
            per[f]["diff_vs_flips0"] = per[f]["diff_ms"] / base
        result["configs"][name] = {"desc": cfg["desc"], "flips": per}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
