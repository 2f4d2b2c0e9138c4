"""Timing of the mesh exporter's texture bake (dreammat_b200/texbake.py) on the mesh bench.py uses.

Input: procedural_mesh(100000, 0.8, 0) with seeded hash-grid parameters, at T = 1024 / 2048 / 4096.
Device stages (CUDA events, median over --reps after --warmup): raster, positions (compaction + interpolation), hash grid,
export + quantise + scatter, fill, and their total.  Host: atlas time and covered-texel fraction.  Comparison leg, on the
host CPU: the reference's padding step, cv2.inpaint(..., padding, INPAINT_TELEA) on the same hole mask.
Prints one JSON line (with the GPU name and power limit); --out also writes it to a file.

    python scripts/bench_export.py --out /tmp/export.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

STAGES = ("raster", "positions", "hashgrid", "export", "fill")


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:          # read-only query; its absence is reported, not guessed
        return f"unavailable ({type(e).__name__})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1024,2048,4096")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--padding", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_export.py measures the device bake: no CUDA device")
    import cv2
    from dreammat_b200 import system as Y
    from dreammat_b200 import texbake as TB
    from dreammat_b200 import uvatlas as U
    from dreammat_b200.scene import procedural_mesh
    v, f = procedural_mesh(100000, 0.8, 0)
    geo = Y.DreamMatMesh(device="cuda", mesh=(v, f))
    g = torch.Generator().manual_seed(0)
    geo.grid.copy_((torch.rand(geo.n_grid, generator=g) * 2 - 1).cuda())
    mat = Y.DreamMatMaterial(device="cuda")
    res = {"gpu": torch.cuda.get_device_name(0), "power_limit": power_limit(), "faces": int(f.shape[0]),
           "padding": a.padding, "reps": a.reps, "sizes": {}}
    for T in (int(s) for s in a.sizes.split(",")):
        t0 = time.perf_counter()
        atlas = U.build_atlas(v.numpy(), f.numpy(), T, a.padding)
        atlas_s = time.perf_counter() - t0
        times = {k: [] for k in STAGES + ("total",)}
        for it in range(a.warmup + a.reps):
            ev = []

            def mark(stage):
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                ev.append((stage, e))
            out = TB.bake_textures(geo, mat, T, a.padding, atlas=atlas, return_debug=True, mark=mark)
            torch.cuda.synchronize()
            if it >= a.warmup:
                for i in range(1, len(ev)):
                    times[ev[i][0]].append(ev[i - 1][1].elapsed_time(ev[i][1]))
                times["total"].append(ev[0][1].elapsed_time(ev[-1][1]))
        mask = out["mask"].view(T, T).cpu().numpy()
        covered = int(mask.sum())
        # CPU leg: the reference pads with Telea inpainting over every hole texel of the same mask
        img = (out["map_Kd"].cpu().numpy() * 255).round().astype(np.uint8)
        holes = (1 - mask).astype(np.uint8) * 255
        t0 = time.perf_counter()
        cv2.inpaint(img, holes, a.padding, cv2.INPAINT_TELEA)
        telea_s = time.perf_counter() - t0
        res["sizes"][str(T)] = {
            "device_ms_median": {k: round(float(np.median(x)), 4) for k, x in times.items()},
            "host_atlas_s": round(atlas_s, 3), "charts": int(atlas.face_chart.max()) + 1,
            "covered_texels": covered, "covered_fraction": round(covered / (T * T), 4),
            "cpu_leg_cv2_inpaint_telea_rgb_s": round(telea_s, 3)}
        del out
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
