#!/usr/bin/env python3
"""bench.py -- benchmark of the photomosaic best-fit path on the BASELINE.json configurations.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload cfg4|cfg2|cfg3|cfg5|...] [--configs all|none]
                    [--dump-outputs DIR]

Headline workload (BASELINE.json configs[3], SURVEY.md section 8d "Config 4"): synthetic 7680x4320 main image x 10,000-image
library of 128x128 tiles, CIEDE2000, square cells 128, detail 100 %, repeat range 8 / addition 500. A "step" is one complete
generateBestFits(): preprocessing, the fused difference-sum kernel over cells x library, the repeat-penalised wavefront
selection, grid back on the host. The same job is sharded over N GPUs (strong scaling); under torchrun every rank is one
process on one GPU.

value   : pixel-differences / second (active, in-bound mask pixels x library images; SURVEY.md 8d metric (i)) with the 8-bit inputs
          already resident in HBM when the timed region starts.
e2e     : the same metric through the reference-shaped API from pinned HOST buffers each step: setMainImage + setLibrary (H2D) +
          generateBestFits + getBestFits (D2H).
configs : the other GPU configurations of BASELINE.json AS SPECIFIED, each with value / e2e / kernel roofline / tie band:
          cfg2 = SampleImages main image (tests/golden/images) x 2,000-image substitute library, CIEDE2000, Cells/Hexagon.mcs @128,
          detail 50 %; cfg3 = 4K x 2,000, CIE76, 64 px cells, 3 size levels; cfg5 = 16K x 20,000, RGB Euclidean, Cells/Puzzle.mcs
          @128, detail 50 %. Cell shapes are read and resized by the PRODUCT (mosaic_mcs_load, CellShape.resized).
roofline: the binding EXECUTED pipe of the difference kernel (FP32 lane-ops or MUFU ops per pixel-difference counted from the
          SASS of the shipped library -- profiles/r2_sass_counts.json, tools/sass_counts.py -- x units / CUDA-event duration,
          against the pipe rates measured live by the in-library micro-benchmark).
The CPU oracle package (the reference's own generator compiled into oracle/_ref) is imported ONLY by the cpu_baseline leg and
by --impl reference; the B200 arm builds everything it needs with the product.
--dump-outputs DIR: after the run, DIR/<workload>_best_fits<step>.npy (float64) holds the best-fit grid of every size step that the
last timed step of each B200 workload returned (getBestFits: library index per cell, -1 outside the grid state). The inputs are
seeded, so two builds run with the same arguments can be compared output for output.
bench.py writes nothing into the source tree (no bytecode either), so it runs from a read-only checkout.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # the modules imported below (package, oracle, tools/) leave no __pycache__ in the tree
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CELLS_DIR = os.path.join(ROOT, "tests", "golden", "cells")
SAMPLE_IMAGE = os.path.join(ROOT, "tests", "golden", "images", "edgar-perez-424673-unsplash.jpg")
DIFF_NAMES = ["RGB_EUCLIDEAN", "CIE76", "CIEDE2000"]

# SURVEY.md section 8(d): algorithmic work per pixel-difference of the REFERENCE formula (ColourDifference.cpp as written)
WORK_REFERENCE_FORMULA = {2: {"flop": 110, "sfu": 27}, 0: {"flop": 9, "sfu": 1}, 1: {"flop": 9, "sfu": 1}}

# dram__bytes_read.sum + dram__bytes_write.sum of the difference kernel, per launch on 1 GPU, from the ncu --set full captures
# committed under profiles/ (not measurable inside an un-profiled run): workload -> (bytes, file)
NCU_TRAFFIC = {
    # both pixel-segment launches of the default plan (2 segments, 32 x 8 super-blocks): 15.8 + 14.8 GB read, 0.28 GB written
    "cfg4": (30600000000 + 280000000, "profiles/r2_raster_sweep.txt (ncu dram__bytes_read.sum + dram__bytes_write.sum; round 1: 132.4 GB)"),
    "cfg5": (32300478000 + 15758592, "profiles/r2_diff_euclid_cfg5.txt (ncu --set full at full size; algorithmic 1.28 GB)"),
}

WORKLOADS = {
    "cfg4": dict(h=4320, w=7680, n_lib=10000, cell=128, detail=100, diff=2, rr=8, ra=500, seed=1004,
                 desc="synthetic 8K (7680x4320) main x 10,000-image library, CIEDE2000, cell 128, detail 100%, repeat 8/500"),
    "cfg4-d50": dict(h=4320, w=7680, n_lib=10000, cell=128, detail=50, diff=2, rr=8, ra=500, seed=1004, desc="config 4 at detail 50%"),
    "cfg4-small": dict(h=1080, w=1920, n_lib=1000, cell=128, detail=100, diff=2, rr=8, ra=500, seed=1004,
                       desc="config 4 scaled down (1920x1080 x 1,000 images) for quick runs"),
    "cfg4-med": dict(h=2160, w=3840, n_lib=2500, cell=128, detail=100, diff=2, rr=8, ra=500, seed=1004,
                     desc="config 4 scaled down (3840x2160 x 2,500 images) for kernel tuning"),
    "cfg2": dict(h=4000, w=5000, n_lib=2000, cell=128, detail=50, diff=2, rr=2, ra=500, seed=1002, shape="Hexagon", photo=True,
                 desc="SampleImages/edgar-perez (5000x4000) main x 2,000-image library cut from it (big-lib.mil is absent from the "
                      "reference checkout), CIEDE2000, Cells/Hexagon.mcs @128 (spacing 96/110, odd-row offset 55, clipped edge cells), "
                      "detail 50%, repeat 2/500"),
    "cfg3": dict(h=2160, w=3840, n_lib=2000, cell=64, detail=100, diff=1, rr=0, ra=0, seed=1003, steps=2,
                 desc="synthetic 4K (3840x2160) main x 2,000-image library, CIE76, 64px cells, 3 size levels (entropy sub-cell split)"),
    "cfg5": dict(h=8640, w=15360, n_lib=20000, cell=128, detail=50, diff=0, rr=0, ra=0, seed=1005, shape="Puzzle",
                 desc="synthetic 16K (15360x8640) main x 20,000-image library, RGB Euclidean, Cells/Puzzle.mcs @128 (spacing 108, "
                      "72% active), detail 50%"),
    "cfg5-square": dict(h=8640, w=15360, n_lib=20000, cell=128, detail=50, diff=0, rr=0, ra=0, seed=1005,
                        desc="config 5 with square cells (round-1 shape of this workload; kernel comparison only)"),
    "cfg5-small": dict(h=2160, w=3840, n_lib=4000, cell=128, detail=50, diff=0, rr=0, ra=0, seed=1005, shape="Puzzle",
                       desc="config 5 scaled down (3840x2160 x 4,000 images) for quick runs"),
}
SECONDARY = ["cfg2", "cfg3", "cfg5"]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--configs", default="all", choices=["all", "none"],
                    help="all: after the headline workload also run BASELINE configs 2, 3 and 5 (a few steps each) into the `configs` object")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=45.0, help="target CPU time of the full-library cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the best-fit grids of the last timed step of every B200 workload to DIR/<workload>_best_fits<step>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        # that arm times the CPU generator on a sample of cells per step, not the whole grid: there is no grid to compare
        ap.error("--dump-outputs writes the B200 arm's best-fit grids; --impl reference computes no whole grid")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, grids_of):
    """grids_of: workload name -> list of best-fit grids (one per size step), written as float64 .npy files (exact for indices)."""
    arrays = {"%s_best_fits%d" % (name, i): g.astype(np.float64) for name, grids in grids_of.items() for i, g in enumerate(grids)}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, "outputs to dump: %d bytes" % total  # a grid has one entry per cell: a few hundred KB at most
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------- shared by both arms (no oracle, no GPU)

def make_inputs(cfg, main_out=None, lib_out=None):
    """Seeded inputs of a workload as numpy arrays (optionally written into caller-provided pinned buffers)."""
    from mosaicmagnifique_b200 import synthetic
    H, W, N, S = cfg["h"], cfg["w"], cfg["n_lib"], cfg["cell"]
    if cfg.get("photo"):
        import cv2  # JPEG decoding of the fixture only (the reference reads it with cv::imread as well)
        main = cv2.imread(SAMPLE_IMAGE, cv2.IMREAD_COLOR)
        assert main is not None and main.shape == (H, W, 3), "tests/golden/images fixture missing"
        lib = synthetic.make_photo_library(main, N, S, cfg["seed"])
    else:
        main = synthetic.make_main_image(H, W, cfg["seed"] + 1000)
        lib = synthetic.make_library(N, S, cfg["seed"], out=lib_out)
    if main_out is not None:
        main_out[...] = main
        main = main_out
    if lib_out is not None and lib is not lib_out:
        lib_out[...] = lib
        lib = lib_out
    return main, lib


def make_shape(cfg):
    """The workload's top-level cell shape, built by the PRODUCT only: square cells, or a .mcs file of the reference read by
    mosaic_mcs_load and resized to the cell size by the library's host model (CellShape::resized)."""
    from mosaicmagnifique_b200 import CellShape, load_mcs
    if cfg.get("shape"):
        return load_mcs(os.path.join(CELLS_DIR, cfg["shape"] + ".mcs")).resized(cfg["cell"])
    return CellShape(cfg["cell"])


def describe(cfg, name, world):
    """`config` of the JSON line: identical in both arms (static description of the workload)."""
    return {"workload": cfg["desc"], "name": name, "main": [cfg["w"], cfg["h"]], "library": cfg["n_lib"], "cell": cfg["cell"],
            "detail": cfg["detail"], "size_steps": cfg.get("steps", 0), "cell_shape": cfg.get("shape", "square"),
            "colour_difference": DIFF_NAMES[cfg["diff"]], "repeat": [cfg["rr"], cfg["ra"]],
            "cache": "packed library + cells of a step exceed the 126 MB L2 many times over; nothing is reused across steps",
            "parallelism": ("valid cells (raster order) sharded over %d GPUs, library replicated, top-K candidates all-gathered (NCCL)" % world)
            if world > 1 else "1 GPU"}


# ----------------------------------------------------------------------------- clocks

class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.proc.wait(timeout=10)
        self.t.join(timeout=2)
        num = lambda s: s.replace(".", "").isdigit()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and num(r[1])]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and num(r[2])]
        pw = [float(r[3]) for r in self.rows if len(r) >= 9 and num(r[3])]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- CPU reference arm / baseline (the ONLY oracle users)

class CpuReference:
    """The reference's CPU generator on bounded samples of a workload, 1 thread (CPUPhotomosaicGenerator is single-threaded),
    f64, early exit on.
    kind "reference": the reference's OWN PhotomosaicGeneratorBase.cpp / CPUPhotomosaicGenerator.cpp / ColourDifference.cpp /
    GridUtility.cpp, compiled unmodified into oracle/_ref/libref_core.so (oracle/Makefile; the prebuilt library travels to the GPU
    box); a timed call is its setGridState + generateBestFits + getBestFits on 8-bit inputs already handed to its setters.
    generateBestFits preprocesses the WHOLE main image and library on every call; at full size that is amortised over thousands
    of cells, in a sample it is not, so it is measured with an empty grid state and subtracted (which only favours the CPU).
    kind "port": the plain-C restatement (oracle/mosaic_oracle.c) when that library is absent or unusable."""

    def __init__(self, cfg, main, lib):
        from oracle import oracle
        self.o = oracle
        self.cfg, self.main, self.lib = cfg, main, lib
        shp = make_shape(cfg)  # product-side reading / resizing of the cell shape, handed to the checker as plain numbers
        osh = oracle.CellShape.from_mask(shp.getCellMask())
        osh.row_spacing, osh.col_spacing = shp.rowSpacing, shp.colSpacing
        osh.alt_row_spacing, osh.alt_col_spacing = shp.alternateRowSpacing, shp.alternateColSpacing
        osh.alt_row_offset, osh.alt_col_offset = shp.alternateRowOffset, shp.alternateColOffset
        osh.alt_col_flip_h, osh.alt_col_flip_v = shp.alternateColFlipHorizontal, shp.alternateColFlipVertical
        osh.alt_row_flip_h, osh.alt_row_flip_v = shp.alternateRowFlipHorizontal, shp.alternateRowFlipVertical
        self.og = oracle.CellGroup.make(osh, cfg["detail"], 0)  # samples are taken on the top size level
        self.state = oracle.grid_state(self.og, main)[0]
        ys, xs = np.nonzero(self.state >= 0)
        self.valid = list(zip(ys.tolist(), xs.tolist()))  # raster order
        self.use_ref = oracle.reference_generator_available()
        self._gens = {}

    def _gen(self, n_lib):
        """a reference generator object holding the first n_lib library images"""
        if n_lib not in self._gens:
            for g in self._gens.values():
                g.close()
            self._gens.clear()
            o, c = self.o, self.cfg
            g = o.ReferenceGenerator(self.main, self.lib[:n_lib], self.og, c["diff"], 0, c["rr"], c["ra"])
            tm = {}
            g.generate([np.full_like(self.state, -1)], tm)  # also the first-touch warm-up of its buffers
            g.generate([np.full_like(self.state, -1)], tm)
            g.fixed_seconds = tm["seconds"]
            self._gens[n_lib] = g
        return self._gens[n_lib]

    def state_of(self, cells):
        st = np.full_like(self.state, -1)
        for y, x in cells:
            st[y, x] = 0
        return st

    def _prepared(self, n_lib):
        o, c = self.o, self.cfg
        if getattr(self, "_prep_n", None) != n_lib:
            self._mains = [o.to_working_space(self.main, c["diff"])]
            self._lib_f = o.preprocess_library(self.lib[:n_lib], self.og, c["diff"])
            self._prep_n = n_lib
        return self._mains, self._lib_f

    def nominal(self, st, n_lib):
        """nominal pixel-diffs of a sample: active (flipped mask) pixels inside each cell's detail-space bound x library images --
        the unit the engine counts (mosaic_timings.pixel_diffs) and the C port reports as `nominal`"""
        o = self.o
        _, bounds, flips, _ = o.extract_cells([np.zeros(self.main.shape, np.float32)], self.og, 0, st)
        m4 = self.og.detail_cells[0].masks4()
        act = 0
        for (bx, by, bw, bh), f in zip(np.asarray(bounds).reshape(-1, 4), np.asarray(flips).ravel()):
            act += int(np.count_nonzero(m4[f][by:by + bh, bx:bx + bw]))
        return act * n_lib

    def counts(self, st, n_lib):
        """nominal / visited pixel-diffs of a sample from the C port's statistics (untimed; same loops, pinned in tests/)"""
        o, c = self.o, self.cfg
        mains, lib_f = self._prepared(n_lib)
        cells, bounds, flips, _ = o.extract_cells(mains, self.og, 0, st)
        r = o.generate_step(c["diff"], cells, bounds, flips, lib_f, self.og.detail_cells[0].masks4(), st, c["rr"], c["ra"],
                            want_D=False, early_exit=True)
        return r.nominal, r.visited

    def timed(self, cells, n_lib):
        """seconds of the best-fit loops for `cells` x the first n_lib images (fixed per-call preprocessing subtracted)"""
        st = self.state_of(cells)
        if self.use_ref:
            try:
                g = self._gen(n_lib)
                tm = {}
                g.generate([st], tm)
                return max(tm["seconds"] - g.fixed_seconds, 1e-9), g.fixed_seconds, "reference"
            except Exception as e:  # noqa: BLE001  -- a library built on another machine may not load / run here
                print("cpu baseline: reference object code unusable here (%s), timing the C port instead" % e, file=sys.stderr)
                self.use_ref = False
        o, c = self.o, self.cfg
        mains = [o.to_working_space(self.main, c["diff"])]
        lib_f = o.preprocess_library(self.lib[:n_lib], self.og, c["diff"])
        cl, bounds, flips, _ = o.extract_cells(mains, self.og, 0, st)
        m4 = self.og.detail_cells[0].masks4()
        t1 = time.perf_counter()
        o.generate_step(c["diff"], cl, bounds, flips, lib_f, m4, st, c["rr"], c["ra"], want_D=False, early_exit=True)
        return time.perf_counter() - t1, 0.0, "port"

    def sample(self, cells, n_lib, what, want_visited=True):
        secs, fixed, kind = self.timed(cells, n_lib)
        st = self.state_of(cells)
        if want_visited:
            nominal, visited = self.counts(st, n_lib)
            assert nominal == self.nominal(st, n_lib)
        else:
            nominal, visited = self.nominal(st, n_lib), None
        return {"seconds": secs, "nominal": nominal, "visited": visited, "kind": kind, "cells": len(cells), "n_lib": n_lib,
                "nominal_per_s": nominal / secs, "visited_per_s": visited / secs if want_visited else None,
                "visited_fraction": visited / max(nominal, 1) if want_visited else None,
                "sample": "%s: %d cell(s) x %s%d library images of the workload, early exit on%s"
                          % (what, len(cells), "all " if n_lib == len(self.lib) else "the first ", n_lib,
                             "; fixed per-call preprocessing of the whole main image and library (%.2f s) subtracted" % fixed
                             if kind == "reference" else "")}

    def close(self):
        for g in self._gens.values():
            g.close()
        self._gens.clear()


CPU_NOTE = {
    "reference": "the reference's own PhotomosaicGeneratorBase.cpp + CPUPhotomosaicGenerator.cpp + ColourDifference.cpp + GridUtility.cpp "
                 "compiled unmodified (oracle/_ref/libref_core.so, recipe oracle/Makefile), OpenCV calls inside them answered by cv2; 1 "
                 "thread because CPUPhotomosaicGenerator is single-threaded; value counts NOMINAL pixel-diffs (what the early exit skips "
                 "is credited), visited_per_s the differences actually evaluated",
    "port": "oracle/mosaic_oracle.c (plain-C restatement; the reference-compiled library oracle/_ref/libref_core.so is absent), 1 thread; "
            "value counts nominal pixel-diffs (early exit credited), visited_per_s the differences actually evaluated",
}


def cpu_baseline(cfg, main, lib, seconds):
    """SURVEY.md 8(d): (A) the first cells of the grid x the FULL library and (B) one grid row x 256 images; A is the headline."""
    ref = CpuReference(cfg, main, lib)
    n_full = len(lib)
    probe_n = min(n_full, 256)
    t_probe, _, _ = ref.timed(ref.valid[:1], probe_n)                      # calibrate: one cell x 256 images
    per_cell_full = t_probe * n_full / probe_n
    k = int(max(1, min(len(ref.valid), seconds / max(per_cell_full, 1e-9))))
    a = ref.sample(ref.valid[:k], n_full, "A")
    row0 = [c for c in ref.valid if c[0] == ref.valid[0][0]]
    b = ref.sample(row0, probe_n, "B (first grid row)")
    ref.close()
    return {"value": a["nominal_per_s"], "unit": "pixel-diffs/s", "cores": 1, "kind": a["kind"], "sample": a["sample"],
            "visited_per_s": a["visited_per_s"], "visited_fraction": a["visited_fraction"], "seconds": a["seconds"],
            "second_sample": {k2: b[k2] for k2 in ("sample", "nominal_per_s", "visited_per_s", "visited_fraction", "seconds")},
            "note": CPU_NOTE[a["kind"]]}


def run_reference(args, name, cfg):
    """--impl reference: every step times the reference's CPU generator on a bounded sample of the workload -- a different cell of
    the first grid row each step x as much of the library as the per-step budget allows (the FULL library when it fits), so that
    the whole --steps/--warmup run ends within a few minutes."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    main, lib = make_inputs(cfg)
    ref = CpuReference(cfg, main, lib)
    n_full = len(lib)
    budget = max(3.0, 240.0 / max(1, args.steps + args.warmup))             # seconds per step
    probe_n = min(n_full, 256)
    t_probe, _, _ = ref.timed(ref.valid[:1], probe_n)
    per_cell_full = t_probe * n_full / probe_n
    if per_cell_full <= budget:
        n_lib, k = n_full, int(max(1, min(8, budget / per_cell_full)))
    else:
        n_lib, k = int(max(probe_n, min(n_full, n_full * budget / per_cell_full))), 1
    cells_of = lambda i: [ref.valid[(i * k + j) % len(ref.valid)] for j in range(k)]
    for i in range(args.warmup):
        ref.timed(cells_of(i), n_lib)
    t0 = time.perf_counter()
    tot_nominal = 0
    tot_s = 0.0
    last = None
    for i in range(args.steps):
        # the evaluated ("visited") share is measured on the last step's sample only: it needs a second, untimed run of the loops
        last = ref.sample(cells_of(args.warmup + i), n_lib, "per step", want_visited=(i == args.steps - 1))
        tot_nominal += last["nominal"]
        tot_s += last["seconds"]
    wall = time.perf_counter() - t0
    ref.close()
    value = tot_nominal / tot_s
    out = {"impl": "reference", "metric": "pixel-diffs/sec", "value": value, "unit": "pixel-diffs/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / args.steps, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": describe(cfg, name, args.gpus),
           "cpu_baseline": {"value": value, "unit": "pixel-diffs/s", "cores": 1, "kind": last["kind"], "sample": last["sample"],
                            "visited_per_s": value * last["visited_fraction"], "visited_fraction": last["visited_fraction"],
                            "note": CPU_NOTE[last["kind"]]},
           "e2e": {"value": value, "unit": "pixel-diffs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0, "wall_s": wall}
    print(json.dumps(out))


# ----------------------------------------------------------------------------- the B200 arm

def sass_counts():
    """Executed work per pixel-difference of the two difference kernels, counted from the SASS of the library by
    tools/sass_counts.py (committed artefact profiles/r2_sass_counts.json + the loop listings next to it). Where cuobjdump exists
    the counts are re-derived from the library that is actually loaded and compared with the artefact."""
    path = os.path.join(ROOT, "profiles", "r2_sass_counts.json")
    d = json.load(open(path))
    check = "not re-derived (cuobjdump unavailable)"
    try:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import contextlib
        import io

        import sass_counts as sc
        from mosaicmagnifique_b200 import library_path
        with contextlib.redirect_stdout(io.StringIO()):
            live = sc.analyse(library_path())
        same = all(live["kernels"][k]["per_pixel_diff"] == d["kernels"][k]["per_pixel_diff"] for k in d["kernels"])
        check = "re-derived from the loaded library with cuobjdump: %s" % ("identical" if same else "DIFFERENT from the artefact (live counts used)")
        if not same:
            d = live
    except Exception as e:  # noqa: BLE001
        check = "not re-derived (%s)" % type(e).__name__
    return d, os.path.relpath(path, ROOT), check


class B200Run:
    """One workload on this rank's GPU through the reference-shaped API."""

    def __init__(self, name, cfg, rank, world, local_rank):
        import torch
        from mosaicmagnifique_b200 import CellGroup, PhotomosaicGenerator
        self.torch = torch
        self.name, self.cfg, self.rank, self.world, self.local_rank = name, cfg, rank, world, local_rank
        H, W, N, S = cfg["h"], cfg["w"], cfg["n_lib"], cfg["cell"]
        # synthetic inputs, identical on every rank (seeded), in PINNED host memory for the e2e leg
        self.main_t = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory()
        self.lib_t = torch.empty((N, S, S, 3), dtype=torch.uint8).pin_memory()
        make_inputs(cfg, self.main_t.numpy(), self.lib_t.numpy())
        self.gen = gen = PhotomosaicGenerator(local_rank)
        cg = CellGroup()
        cg.setCellShape(make_shape(cfg))
        cg.setDetail(cfg["detail"])
        cg.setSizeSteps(cfg.get("steps", 0))
        gen.setColourDifference(cfg["diff"])
        gen.setCellGroup(cg)
        gen.setRepeat(cfg["rr"], cfg["ra"])
        self.h2d_lib = self.lib_t.numel()
        self.h2d_main = self.main_t.numel()
        self.load_inputs(first=True)
        self.state = gen.computeGridState()
        self.valid_cells = int(sum((s >= 0).sum() for s in self.state))

    def load_inputs(self, first=False):
        from mosaicmagnifique_b200.parallel import set_library_sharded, set_main_image_sharded
        gen, cfg = self.gen, self.cfg
        H, W, N, S = cfg["h"], cfg["w"], cfg["n_lib"], cfg["cell"]
        if self.world > 1:
            # every rank uploads only what it computes on: 1/world of the library over PCIe (reduced to the detail size on the GPU,
            # the rest arrives over NVLink, one in-place NCCL all-gather) and the main-image rows its cells read. The grid state is
            # an input of generateBestFits (setGridState), so the rows are known before the upload; the very first load brings the
            # whole image because computeGridState's entropy rule reads all of it.
            self.h2d_lib = set_library_sharded(gen, self.lib_t, self.rank, self.world)
            if first:
                gen.setMainImagePtr(self.main_t.data_ptr(), H, W, W * 3)
            else:
                gen.setGridState(self.state)
                gen.setShard(self.rank, self.world)
                self.h2d_main = set_main_image_sharded(gen, self.main_t)
        else:
            gen.setMainImagePtr(self.main_t.data_ptr(), H, W, W * 3)
            gen.setLibraryPtr(self.lib_t.data_ptr(), N, S)

    def step(self):
        from mosaicmagnifique_b200.parallel import generate_sharded
        gen = self.gen
        gen.setGridState(self.state)
        if self.world > 1:
            grids, _ = generate_sharded(gen, self.rank, self.world)
        else:
            assert gen.generateBestFits()
            grids = gen.getBestFits()
        return grids

    def barrier(self):
        torch = self.torch
        torch.cuda.synchronize()
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def allmax(self, vals):
        if self.world == 1:
            return list(vals)
        t = self.torch.tensor(list(vals), device="cuda", dtype=self.torch.float64)
        self.torch.distributed.all_reduce(t, op=self.torch.distributed.ReduceOp.MAX)
        return t.tolist()

    def measure(self, steps, warmup, e2e_steps, sample_clocks):
        gen = self.gen
        for _ in range(warmup):
            grids = self.step()
        clocks = ClockSampler(self.local_rank) if sample_clocks else None
        self.barrier()
        if clocks:
            clocks.start()
        t0 = time.perf_counter()
        phase = {"preprocess_ms": 0.0, "diff_ms": 0.0, "select_ms": 0.0}
        launches = 0
        for _ in range(steps):
            grids = self.step()
            tm = gen.getTimings()
            for k in phase:
                phase[k] += tm[k]
            launches += tm["kernel_launches"]
        self.barrier()
        elapsed = time.perf_counter() - t0
        timed_grids = grids
        clk = clocks.stop() if clocks else None
        pixel_diffs = tm["pixel_diffs"]  # whole job (every rank counts all cells of the step)
        local_share = 1.0
        if self.world > 1:
            info = gen.candidateInfo(0)
            local_share = info["n_cells"] / max(1, info["n_valid"])
        elapsed, phase["diff_ms"], phase["preprocess_ms"], phase["select_ms"] = self.allmax(
            [elapsed, phase["diff_ms"], phase["preprocess_ms"], phase["select_ms"]])

        # ---- end-to-end leg: pinned host buffers in, grid out, every step
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            self.load_inputs()
            grids = self.step()
            checksum = int(sum(int(g.sum()) for g in grids))  # touch the D2H result
        self.barrier()
        (e2e_elapsed,) = self.allmax([time.perf_counter() - t0])
        return {"elapsed": elapsed, "steps": steps, "phase": phase, "launches": int(launches), "pixel_diffs": pixel_diffs,
                "pixel_diffs_nominal": tm["pixel_diffs_nominal"], "local_share": local_share, "clocks": clk, "e2e_elapsed": e2e_elapsed,
                "e2e_steps": e2e_steps, "checksum": checksum, "h2d": int(self.h2d_main + self.h2d_lib),
                "d2h": int(sum(g.size * 8 for g in grids)), "grids": timed_grids}

    def tie_band(self):
        """cells whose best two penalised candidates are within an FP32-explainable tolerance (untimed, 1 GPU)"""
        gen = self.gen
        gen.setReportMargins(True)
        gen.setGridState(self.state)
        assert gen.generateBestFits()
        rel = []
        for stp in range(len(self.state)):
            b, s2 = gen.getMargins(stp)
            rel.append((s2.astype(np.float64) - b) / np.maximum(b.astype(np.float64), 1e-30))
        gen.setReportMargins(False)
        rel = np.concatenate(rel) if rel else np.zeros(0)
        return {"of": int(rel.size), "cells_within": {"1e-4": int((rel <= 1e-4).sum()), "1e-5": int((rel <= 1e-5).sum()),
                                                      "1e-6": int((rel <= 1e-6).sum())},
                "tolerance_relative": 1e-5, "cells": int((rel <= 1e-5).sum()),
                "note": "cells whose best and second-best penalised scores differ by <= tol relative: only there may the FP32 engine and "
                        "the f64 reference legitimately pick different images (tests/helpers/parity.py uses 1e-5)"}

    def close(self):
        self.gen.close()
        del self.main_t, self.lib_t


def roofline_of(name, cfg, m, mb, peaks, sass, world):
    """Roofline of the workload's difference kernel from live numbers: executed pipe work (SASS counts) / CUDA-event duration."""
    kern = "diff_sum" if cfg["diff"] == 2 else "diff_euclid"
    per = sass[0]["kernels"][kern]["per_pixel_diff"]
    diff_s = m["phase"]["diff_ms"] * 1e-3 / m["steps"]          # all diff launches of one step on the slowest rank (CUDA events)
    units = m["pixel_diffs"] * m["local_share"]                  # pixel-diffs those launches process on one GPU
    fp32_rate, mufu_rate = per["fp32_lane_ops"] * units / diff_s, per["mufu"] * units / diff_s
    f_fp32, f_mufu = fp32_rate / mb[1], mufu_rate / mb[2]
    work = WORK_REFERENCE_FORMULA[cfg["diff"]]
    N = cfg["n_lib"]
    out = {"kernel": kern + "_kernel", "kernel_ms": diff_s * 1e3, "launches_per_step": 1 + cfg.get("steps", 0),
           "bound": "fp32-pipe" if f_fp32 >= f_mufu else "mufu-pipe",
           "achieved": (fp32_rate if f_fp32 >= f_mufu else mufu_rate) / 1e12,
           "peak": (mb[1] if f_fp32 >= f_mufu else mb[2]) / 1e12,
           "unit": "T lane-op/s" if f_fp32 >= f_mufu else "T MUFU-op/s",
           "frac": max(f_fp32, f_mufu),
           "executed_fp32": {"lane_ops_per_pixel_diff": per["fp32_lane_ops"], "achieved_per_s": fp32_rate, "peak_per_s": mb[1], "frac": f_fp32},
           "executed_mufu": {"ops_per_pixel_diff": per["mufu"], "achieved_per_s": mufu_rate, "peak_per_s": mb[2], "frac": f_mufu},
           "counts_source": "%s (cuobjdump -sass loop body of the shipped library, tools/sass_counts.py; %s)" % (sass[1], sass[2]),
           "peak_source": "live in-library micro-benchmark (FFMA2 lane-ops/s, MUFU.RSQ ops/s) on this GPU at its current clocks",
           "pixel_diffs_per_s_kernel": units / diff_s,
           "frac_reference_formula": work["sfu"] * units / diff_s / mb[2],
           "reference_formula_note": "SURVEY 8d counts the REFERENCE formula (%d flop + %d special-function ops per pixel-diff); the kernel's "
                                     "algebra executes fewer, so this ratio is not a pipe utilisation and may exceed 1" % (work["flop"], work["sfu"]),
           "traffic": NCU_TRAFFIC[name][0] if (world == 1 and name in NCU_TRAFFIC) else None,
           "traffic_source": NCU_TRAFFIC[name][1] if (world == 1 and name in NCU_TRAFFIC) else None}
    if cfg["diff"] == 2:
        out["mixed_pipe_ceiling_pixel_diffs_per_s"] = mb[6]
    # secondary bound: bytes the launch must move at least once (packed library + packed cells of the top level)
    ds = int(cfg["cell"] * cfg["detail"] / 100)
    lib_b, cell_b = (16, 20) if cfg["diff"] == 2 else (12, 16)
    act = m["pixel_diffs"] / max(m["pixel_diffs_nominal"], 1)    # active share of the detail cell (mask + bounds)
    min_bytes = (N * lib_b + m["valid_cells"] * m["local_share"] * cell_b) * ds * ds * min(1.0, act * 1.02)
    out["hbm"] = {"min_bytes_per_step": min_bytes, "achieved_gbs": min_bytes / diff_s / 1e9, "peak_gbs": peaks.get("hbm_gbs"),
                  "frac": (min_bytes / diff_s / 1e9) / peaks["hbm_gbs"] if peaks.get("hbm_gbs") else None,
                  "peak_source": "MEASURED_PEAKS.json" if peaks else "absent"}
    return out


def summarise(name, cfg, m, world, roof):
    sec = m["elapsed"] / m["steps"]
    return {"config": describe(cfg, name, world), "value": m["pixel_diffs"] / sec, "unit": "pixel-diffs/s", "generate_ms": 1e3 * sec,
            "steps": m["steps"], "valid_cells": m["valid_cells"], "pixel_diffs_per_step": m["pixel_diffs"],
            "phases_ms_per_step": {k: v / m["steps"] for k, v in m["phase"].items()},
            "e2e": {"value": m["pixel_diffs"] / (m["e2e_elapsed"] / m["e2e_steps"]), "unit": "pixel-diffs/s",
                    "ms_per_step": 1e3 * m["e2e_elapsed"] / m["e2e_steps"], "steps": m["e2e_steps"], "h2d_bytes_per_step": m["h2d"],
                    "d2h_bytes_per_step": m["d2h"], "result_checksum": m["checksum"]},
            "gpu_launches": m["launches"], "roofline": roof}


def main():
    args = parse()
    cfg = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, args.workload, cfg)
        return

    import ctypes

    import torch
    import torch.distributed as dist

    from mosaicmagnifique_b200 import capi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import datetime
        # a collective that does not complete within 5 minutes is a bug, not a slow step: fail fast instead of holding 8 GPUs
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=300))

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peaks = json.load(open(peaks_path)) if os.path.exists(peaks_path) else {}
    sass = sass_counts()

    # ---- headline workload
    run = B200Run(args.workload, cfg, rank, world, local_rank)
    m = run.measure(args.steps, args.warmup, max(1, min(args.steps, 3)), sample_clocks=True)
    m["valid_cells"] = run.valid_cells
    outputs = {args.workload: m["grids"]}
    mb = np.zeros(12)
    capi().mosaic_kernel_microbench(local_rank, mb.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), 12)
    head = summarise(args.workload, cfg, m, world, roofline_of(args.workload, cfg, m, mb, peaks, sass, world))
    tie = run.tie_band() if world == 1 else None
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(cfg, run.main_t.numpy(), run.lib_t.numpy(), args.cpu_seconds)
    run.close()
    del run
    torch.cuda.empty_cache()

    # ---- the other BASELINE configurations, a few steps each
    configs = {}
    if args.configs == "all" and args.workload == "cfg4":
        for name in SECONDARY:
            c2 = WORKLOADS[name]
            r2 = B200Run(name, c2, rank, world, local_rank)
            # short steps after a long idle phase (input generation on the CPU): warm up for >= 0.5 s so that the clocks are up.
            # The number of warm-up steps comes from a timing, so it is agreed on by ALL ranks (max over ranks) -- every step is a
            # collective under torchrun, and ranks that disagree on the count dead-lock.
            t_w = time.perf_counter()
            r2.step()
            (one,) = r2.allmax([max(time.perf_counter() - t_w, 1e-3)])
            m2 = r2.measure(min(args.steps, 5), max(3, min(50, int(0.5 / one))), 2, sample_clocks=True)
            m2["valid_cells"] = r2.valid_cells
            outputs[name] = m2["grids"]
            s2 = summarise(name, c2, m2, world, roofline_of(name, c2, m2, mb, peaks, sass, world))
            s2["clocks"] = m2["clocks"]
            if world == 1:
                s2["tie_band"] = r2.tie_band()
            configs[name] = s2
            r2.close()
            del r2
            torch.cuda.empty_cache()

    if rank == 0:
        out = {"metric": "pixel-diffs/sec", "value": head["value"], "unit": "pixel-diffs/s", "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": head["generate_ms"], "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": head["config"], "generate_ms": head["generate_ms"],
               "valid_cells": head["valid_cells"], "pixel_diffs_per_step": head["pixel_diffs_per_step"],
               "phases_ms_per_step": head["phases_ms_per_step"], "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
               "clocks": m["clocks"], "roofline": head["roofline"],
               "microbench": {"ffma_lane_ops_per_s": mb[0], "ffma2_lane_ops_per_s": mb[1], "mufu_rsq_per_s": mb[2], "mufu_ex2_per_s": mb[3],
                              "sm_count": int(mb[4]), "ciede_mix_pairs_per_s": mb[6], "ffma2_plus_ffma_lane_ops_per_s": [mb[9], mb[10]]}}
        if tie is not None:
            out["tie_band"] = tie
        if cpu is not None:
            out["cpu_baseline"] = cpu
        if configs:
            out["configs"] = configs
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
