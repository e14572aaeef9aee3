"""Multiplet emissions on the 100x60 grid (24 x 16 rays): influence build, LU against GMRES on one GPU, and the whole
source function through one handle over 1 and over every visible GPU.

    python tools/mult_large.py --out DIR [--kinds 0,1] [--shape 100,60,24,16] [--repeats 3]

For each kind (0 = O I 102.6 nm, 1 = H Lyman multiplet) it writes DIR/mult_large.json: device name and power limit
(nvidia-smi, read-only queries), the build's traversal and march times and ray-voxel steps per second, the solve with
B200RT_SOLVER=lu and =gmres on device 0 (device time of the solve phase, host time around the synchronising call, GMRES
steps, true residuals, max |S_gmres - S_lu| / max |S_lu|), and b200rt_generate_S through a handle over 1 and over all
visible devices (host time; the distributed solve where the grid takes it).  Repeats after one warm-up; the median is
reported.  Needs a CUDA device: there is no fallback."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import importlib  # noqa: E402

synth = importlib.import_module("3d_planetary_rt_model_b200.synth")
binding = importlib.import_module("3d_planetary_rt_model_b200.binding")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout
    return [dict(zip(("index", "name", "power_limit", "max_sm_clock"), (x.strip() for x in line.split(","))))
            for line in q.strip().splitlines()]


def timed(fn, repeats):
    fn()                                             # warm-up: module load, allocations, shared-memory limits
    out = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        r = fn()
        out.append((time.perf_counter() - t0, r))
    return out


def med(xs):
    return float(np.median(xs))


def solve_with(G, solver, repeats):
    os.environ["B200RT_SOLVER"] = solver
    try:
        runs = timed(lambda: (G.solve(), G.ctx.kernel_ms(binding.PH_SOLVE), G.last_solve_steps()), repeats)
    finally:
        del os.environ["B200RT_SOLVER"]
    res = runs[-1][1]
    return dict(host_ms=med([t * 1e3 for t, _ in runs]), device_ms=med([r[1][0] for _, r in runs]),
                launches=res[1][1], gmres_steps=res[2] if solver == "gmres" else None,
                residual=G.ctx.residual(0)), G.vectors()["S"].copy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--kinds", default="0,1")
    ap.add_argument("--shape", default="100,60,24,16")
    ap.add_argument("--repeats", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    shape = tuple(int(x) for x in a.shape.split(","))
    n_dev = binding.load().b200rt_device_count()
    if n_dev < 1:
        raise SystemExit("no CUDA device")
    report = dict(gpus=gpu_info(), visible_devices=n_dev, shape=shape, kinds={})
    for kind in (int(k) for k in a.kinds.split(",")):
        scn = synth.make_multiplet_scenario(kind, *shape, sza_T_contrast=0.1)
        G = binding.GpuMultiplet(scn, "f64", device=0)
        r = dict(n_vox=scn.n_vox, n_upper=G.n_upper, n_el=G.n_el, K_bytes=G.n_el * G.n_el * 8)
        builds = timed(lambda: (G.build_rows(), G.ctx.kernel_ms(binding.PH_TRAVERSE)[0],
                                G.ctx.kernel_ms(binding.PH_INFLUENCE)[0]), a.repeats)
        steps = builds[-1][1][0][1]
        march_ms = med([b[2] for _, b in builds])
        r["build"] = dict(host_ms=med([t * 1e3 for t, _ in builds]), traverse_ms=med([b[1] for _, b in builds]),
                          march_ms=march_ms, ray_voxel_steps=steps, steps_per_s=steps / (march_ms * 1e-3))
        r["lu"], S_lu = solve_with(G, "lu", a.repeats)
        r["gmres"], S_gm = solve_with(G, "gmres", a.repeats)
        r["gmres"]["max_diff_vs_lu"] = float(np.abs(S_gm - S_lu).max() / np.abs(S_lu).max())
        del G
        r["generate_S"] = {}
        for n in sorted({1, n_dev}):
            H = binding.GpuMultiplet(scn, "f64", devices=list(range(n)))
            runs = timed(lambda: (H.ctx.generate_S(), H.ctx.kernel_ms(binding.PH_SOLVE), H.last_solve_steps()), a.repeats)
            S = H.vectors()["S"]
            r["generate_S"][str(n)] = dict(host_ms=med([t * 1e3 for t, _ in runs]),
                                           solve_device_ms=med([x[1][0] for _, x in runs]), solve_launches=runs[-1][1][1][1],
                                           gmres_steps=runs[-1][1][2], residual=H.ctx.residual(0),
                                           max_diff_vs_lu=float(np.abs(S - S_lu).max() / np.abs(S_lu).max()))
            del H
        report["kinds"][str(kind)] = r
        print(json.dumps({kind: r}), flush=True)
    with open(os.path.join(a.out, "mult_large.json"), "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
