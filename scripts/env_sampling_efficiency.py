"""Efficiency of environment sampling (RRS_FLAG_ENV_SAMPLING) against the plain render.

For each scene: a flag-off reference at `--ref-mult` times the samples, then `--reps` renders with and without the
flag at equal spp (different seeds).  Reports device time per sample (CUDA events, rrs_stats device_ms), the MSE
against the reference (it includes the reference's own variance, about 1/ref-mult of the flag-off MSE), and the figure
of merit 1 / (MSE * time).  Prints one JSON line per scene and the GPU it ran on.

    python scripts/env_sampling_efficiency.py [--out env_sampling_efficiency.log]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from rayrs_b200 import api, scenes  # noqa: E402


def gpu_info() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # the numbers are still valid; say that the card could not be read
        return f"unknown ({e})"


def measure(name, spec, hdri, spp, reps, ref_mult):
    sc = spec.scene(hdri)
    cam = spec.camera()
    mb = spec.max_bounces
    api.render_gpu(cam, sc, spp, mb)                                   # warm-up: module load, queue allocation
    api.render_gpu(cam, sc, spp, mb, flags=api.RRS_FLAG_ENV_SAMPLING)
    ref = np.zeros((cam.y_pixels(), cam.x_pixels(), 3))
    for k in range(ref_mult):
        ref += api.render_gpu(cam, sc, spp, mb, seed=10_000 + k)
    ref /= ref_mult
    res = {"scene": name, "width": cam.x_pixels(), "height": cam.y_pixels(), "spp": spp, "max_bounces": mb,
           "reps": reps, "ref_spp": spp * ref_mult}
    for tag, flags in (("off", 0), ("on", api.RRS_FLAG_ENV_SAMPLING)):
        mse, ms, rays = [], [], []
        for r in range(reps):
            img = api.render_gpu(cam, sc, spp, mb, seed=20_000 + r, flags=flags).astype(np.float64)
            st = sc.stats()
            assert st["census_mismatch_pixels"] == 0 and st["nan_pixels"] == 0
            mse.append(float(np.mean((img - ref) ** 2)))
            ms.append(st["device_ms"])
            rays.append(st["rays"])
        t = float(np.median(ms)) / spp
        m = float(np.mean(mse))
        res[tag] = {"mse": m, "ms_per_sample": t, "rays_per_path": float(np.mean(rays)) / (cam.x_pixels() * cam.y_pixels() * spp),
                    "fom": 1.0 / (m * t), "ms_spread": [float(min(ms)), float(max(ms))]}
    res["fom_ratio"] = res["on"]["fom"] / res["off"]["fom"]
    res["mse_ratio"] = res["off"]["mse"] / res["on"]["mse"]
    res["time_ratio"] = res["on"]["ms_per_sample"] / res["off"]["ms_per_sample"]
    sc.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ref-mult", type=int, default=64)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    lines = [f"gpu: {gpu_info()}"]
    print(lines[0], flush=True)
    c1 = scenes.CONFIGS["c1"]
    runs = [("c1 diffuse_single_sphere, synthetic_hdri 2048x1024 (sun clipped to 3)", c1.specs()[0],
             scenes.synthetic_hdri(2048, 1024), c1.spp),
            ("sun_spheres 512x384, sun_hdri 1024x512 (unclipped sun, 2000x the sky)", scenes.sun_spheres(512, 384),
             scenes.sun_hdri(1024, 512), 64)]
    for name, spec, hdri, spp in runs:
        res = measure(name, spec, hdri, spp, a.reps, a.ref_mult)
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
