"""Cost of the scaled build (mosaic_build_photomosaic_scaled) on BASELINE configs 4 and 5 at full size.

For each config: two generates (host clock; the second is reported beside the builds), then builds at k = 1, 2 and 4 from a
render library that is the matching library upsampled by nearest neighbour on the GPU (what the build reads does not depend on the
pixel values), into
  * device memory (the kernels alone: owner scatter and gather),
  * pinned host memory (device bands copied out with cudaMemcpy2DAsync),
  * pageable host memory.
Every time is the median of --rounds builds after one warm-up build, from a host clock around the call (it ends in a stream
synchronise). The gather's bytes are the output plus one read of every covered output pixel's tile pixel (3 bytes) plus the owner map
(8 bytes per main-image pixel); bytes over the build time is reported as GB/s. The GPU name and power limit are read in the same run.

    python tools/bench_render_scale.py [--rounds 5] [--configs cfg4,cfg5] [--scales 1,2,4] [--out FILE]
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


def timed(fn, rounds):
    fn()  # warm-up: first launch, first touch of a pageable buffer
    ts = []
    for _ in range(rounds):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), [round(t, 3) for t in ts]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--configs", default="cfg4,cfg5")
    ap.add_argument("--scales", default="1,2,4")
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch

    import bench
    from mosaicmagnifique_b200 import CellGroup, PhotomosaicGenerator
    dev = torch.device("cuda", 0)
    bg = (0, 0, 0, 0)  # tiles have alpha 255, so the covered pixels are counted from the device output
    result = {"gpu": gpu_info(), "rounds": args.rounds, "configs": {}}
    for name in args.configs.split(","):
        cfg = bench.WORKLOADS[name]
        main_img, lib = bench.make_inputs(cfg)
        H, W = main_img.shape[:2]
        N, S = len(lib), cfg["cell"]
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
        generate_ms = []  # the first generate of the process, then a second one
        for _ in range(2):
            t0 = time.perf_counter()
            assert gen.generateBestFits()
            generate_ms.append((time.perf_counter() - t0) * 1e3)
        lib_t = torch.from_numpy(lib).to(dev)
        per = {}
        for k in (int(v) for v in args.scales.split(",")):
            render = lib_t.repeat_interleave(k, 1).repeat_interleave(k, 2).contiguous() if k > 1 else lib_t
            torch.cuda.synchronize()  # the handle copies on its own stream, which does not wait for torch's
            gen.setRenderLibraryPtr(render.data_ptr(), N, k * S)
            del render
            torch.cuda.empty_cache()
            rows, cols = k * H, k * W
            out_bytes = rows * cols * 4
            entry = {"output": [rows, cols], "output_bytes": out_bytes, "render_library_bytes": N * (k * S) ** 2 * 3}
            out = torch.empty((rows, cols, 4), dtype=torch.uint8, device=dev)
            gen.buildPhotomosaicScaled(bg, out=out)
            covered = int((out[..., 3] == 255).sum().item())
            gather_bytes = out_bytes + 3 * covered + 8 * H * W
            entry.update({"covered_pixels": covered, "gather_bytes": gather_bytes})
            ms, all_ms = timed(lambda: gen.buildPhotomosaicScaled(bg, out=out), args.rounds)
            entry["device"] = {"build_ms": ms, "all_ms": all_ms, "gather_GBps": gather_bytes / ms / 1e6}
            del out
            torch.cuda.empty_cache()
            host = torch.empty((rows, cols, 4), dtype=torch.uint8, pin_memory=True)
            ms, all_ms = timed(lambda: gen.buildPhotomosaicScaled(bg, out=host), args.rounds)
            entry["pinned"] = {"build_ms": ms, "all_ms": all_ms, "output_GBps": out_bytes / ms / 1e6}
            del host
            host = np.empty((rows, cols, 4), np.uint8)
            ms, all_ms = timed(lambda: gen.buildPhotomosaicScaled(bg, out=host), args.rounds)
            entry["pageable"] = {"build_ms": ms, "all_ms": all_ms, "output_GBps": out_bytes / ms / 1e6}
            del host
            per[str(k)] = entry
            print(name, k, json.dumps({m: entry[m]["build_ms"] for m in ("device", "pinned", "pageable")}), flush=True)
        gen.setRenderLibrary(None)
        gen.close()
        del lib_t
        torch.cuda.empty_cache()
        result["configs"][name] = {"desc": cfg["desc"], "generate_ms": generate_ms[1], "first_generate_ms": generate_ms[0],
                                   "main": [H, W], "images": N, "cell": S, "scales": per}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
