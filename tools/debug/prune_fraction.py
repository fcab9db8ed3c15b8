"""Executed share of the CIEDE2000 difference work under exact pruning, for bench.py's workloads (all cells of the step).

    python tools/debug/prune_fraction.py [cfg4 cfg2 ...]

Prints, per workload, evaluated_pixel_diffs / pixel_diffs of one generate (mosaic_timings): the (row, chunk) work the segment
passes executed over the work a complete D needs, and the generate time with and without pruning (setKeepDifferences)."""
import os
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))

import bench  # noqa: E402
from mosaicmagnifique_b200 import CellGroup, PhotomosaicGenerator  # noqa: E402


def main(names):
    for name in names:
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
        gen.setRepeat(cfg["rr"], cfg["ra"])
        state = gen.computeGridState()
        out = {}
        for keep in (False, True, False):
            gen.setGridState(state)
            gen.setKeepDifferences(keep)
            t0 = time.perf_counter()
            assert gen.generateBestFits()
            out[keep] = (time.perf_counter() - t0, gen.getTimings())
        gen.close()
        tm = out[False][1]
        print("%s: cells %d, evaluated / nominal %.4f, generate %.1f ms pruned / %.1f ms complete D" % (
            name, int(sum((s >= 0).sum() for s in state)), tm["evaluated_pixel_diffs"] / tm["pixel_diffs"],
            1e3 * out[False][0], 1e3 * out[True][0]), flush=True)


if __name__ == "__main__":
    main(sys.argv[1:] or ["cfg4", "cfg2"])
