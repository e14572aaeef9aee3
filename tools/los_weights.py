"""Line-of-sight weighting functions (b200rt_los_weights*, DESIGN.md section 4) on the bench workload.

    python tools/los_weights.py --out profiles/r05_los_weights.json [--n-los 1000000] [--repeats 3]

The 100x60 grid with 24x16 rays and bench.py's seeded 10^6 lines of sight, in double and float, with one emission
(bench.py's) and with two (Ly alpha + Ly beta, the facade's).  For each: nnz, the mean and maximum row length and the
device bytes of the matrix; the build (traversal + structure passes + ordering + value pass) and the brightness march
(b200rt_brightness_resident: traversal + ordering + march) on the same resident lines of sight, alternated `repeats`
times after one warm-up of each (medians of device-event times); the products W x and W^T r (device time of the product
kernel, medians over 10 calls) with their compulsory bytes against the HBM bandwidth measured in the same run (a 4 GiB
device-to-device copy, 8 GiB moved; the matrix is larger than the 126 MB L2); and max |W S - brightness| / max
brightness with W S from b200rt_los_weights_apply.  The card's name and power limit are read in the same run
(nvidia-smi, read-only queries).  Needs a CUDA device: there is no fallback."""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
synth = importlib.import_module("3d_planetary_rt_model_b200.synth")
binding = importlib.import_module("3d_planetary_rt_model_b200.binding")
GRID = (100, 60, 24, 16)      # bench.py's grid


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout
    return [dict(zip(("index", "name", "power_limit", "max_sm_clock"), (x.strip() for x in line.split(","))))
            for line in q.strip().splitlines()]


def hbm_peak_gbs(reps=10):
    """bytes read + written by a 4 GiB device-to-device copy over its device time"""
    import torch
    a = torch.empty(1 << 29, dtype=torch.float64, device="cuda:0")
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    gbs = 2 * a.numel() * 8 * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del a, b
    torch.cuda.empty_cache()
    return gbs


def phases(ctx, ids):
    return {p: ctx.kernel_ms(p)[0] for p in ids}


def run(scn, locs, dirs, prec, n_em, repeats, hbm):
    G = binding.GpuModel(scn, prec)
    c = G.ctx
    rng = np.random.default_rng(7)
    S = [rng.uniform(0.5, 1.5, G.n_vox) for _ in range(n_em)]
    for e in range(n_em):
        G.set_sourcefn(e, S[e])
    c.los_upload(c.los_from_MSO(locs, dirs))
    nnz = c.los_weights(10)                         # warm-up of both
    c.brightness_resident(10)
    build, bright = [], []
    build_ph, bright_ph = [], []
    for _ in range(repeats):
        c.los_weights(10)
        ph = phases(c, (binding.PH_TRAVERSE, binding.PH_ORDER, binding.PH_LW_STRUCTURE, binding.PH_LW_VALUES))
        build.append(sum(ph.values()))
        build_ph.append(ph)
        sub_w = c.last_substep_count()
        c.brightness_resident(10)
        ph = phases(c, (binding.PH_TRAVERSE, binding.PH_ORDER, binding.PH_BRIGHTNESS))
        bright.append(sum(ph.values()))
        bright_ph.append(ph)
        sub_b = c.last_substep_count()
    med = lambda v: float(np.median(v))
    out = c.los_download()["brightness"]
    indptr = np.zeros(len(locs) + 1, np.int64)
    c._ck(c.lib.b200rt_los_weights_download(c.h, binding._ptr(indptr), None, None))
    rows = np.diff(indptr)
    real = 8 if prec == "f64" else 4
    n = len(locs)
    r = dict(prec=prec, n_emissions=n_em, n_los=n, nnz=int(nnz), row_len_mean=float(rows.mean()),
             row_len_max=int(rows.max()), empty_rows=int((rows == 0).sum()),
             matrix_device_bytes=int(8 * (n + 1) + 4 * nnz + real * n_em * nnz),
             substeps_build=int(sub_w), substeps_brightness=int(sub_b),
             build_ms=med(build), brightness_ms=med(bright), build_over_brightness=med(build) / med(bright),
             build_ms_all=build, brightness_ms_all=bright,
             build_phases_ms={k: med([p[k] for p in build_ph]) for k in build_ph[0]},
             brightness_phases_ms={k: med([p[k] for p in bright_ph]) for k in bright_ph[0]})
    r["build_phases_ms"] = {name: r["build_phases_ms"][k] for k, name in
                            ((binding.PH_TRAVERSE, "traverse"), (binding.PH_ORDER, "order"),
                             (binding.PH_LW_STRUCTURE, "structure"), (binding.PH_LW_VALUES, "values"))}
    r["brightness_phases_ms"] = {name: r["brightness_phases_ms"][k] for k, name in
                                 ((binding.PH_TRAVERSE, "traverse"), (binding.PH_ORDER, "order"),
                                  (binding.PH_BRIGHTNESS, "march"))}
    # products: compulsory bytes = row_ptr + col + val (+ the dense operands: x gathers hit L2, counted once)
    x, rl = rng.uniform(0, 1, G.n_vox), rng.uniform(0, 1, n)
    prod = {}
    for tr, name, vec in ((0, "W_x", x), (1, "WT_r", rl)):
        c.los_weights_apply(0, vec, bool(tr))
        t = []
        for _ in range(10):
            c.los_weights_apply(0, vec, bool(tr))
            t.append(c.kernel_ms(binding.PH_LW_APPLY)[0])
        byts = 8 * (n + 1) + (4 + real) * nnz + 8 * n + 8 * G.n_vox
        ms = med(t)
        prod[name] = dict(ms=ms, bytes=int(byts), gbs=byts / (ms * 1e-3) / 1e9, hbm_fraction=byts / (ms * 1e-3) / 1e9 / hbm)
    r["products"] = prod
    err = 0.0
    for e in range(n_em):
        WS = c.los_weights_apply(e, S[e])
        err = max(err, float(np.abs(WS - out[e]).max() / np.abs(out[e]).max()))
    r["max_rel_WS_minus_brightness"] = err
    c.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n-los", type=int, default=1000000)
    ap.add_argument("--repeats", type=int, default=3)
    a = ap.parse_args()
    if binding.load().b200rt_device_count() < 1:
        raise SystemExit("no CUDA device")
    hbm = hbm_peak_gbs()
    report = dict(gpus=gpu_info(), grid=list(GRID), n_subsamples=10, hbm_copy_gbs=hbm,
                  guideline="build W in no more than twice the brightness march on the same lines of sight",
                  runs=[])
    locs, dirs = synth.random_los(a.n_los)            # bench.py's seeded set
    for n_em in (1, 2):
        scn = synth.make_scenario(*GRID, n_em=n_em, rmethod=synth.RMETHOD_ALTITUDE, rmax=synth.rMars + 50000e5)
        for prec in ("f64", "f32"):
            r = run(scn, locs, dirs, prec, n_em, a.repeats, hbm)
            print(json.dumps(r), flush=True)
            report["runs"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
