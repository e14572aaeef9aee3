"""Mirror-pair fold of the voxel-origin rays in the influence builds (grid_host.cpp fold_pairs, DESIGN.md section 4).

    python tools/ray_fold.py cpu [--big]                    # the premise on the CPU oracle, double and float
    python tools/ray_fold.py gpu --out DIR [--repeats 3]    # counts and build times on the 100x60 grid

cpu: the rays marched per voxel for n_phi from 6 to 512 (24 polar angles, both precisions: a fold lost to the cos(phi)
tolerance shows up here), then for every voxel and every pair of rays phi_j, phi_(n_phi-1-j) of the 12x8x5x6, 20x12x6x8
and 40x20x7x12 grids (--big: also the 100x60x24x16 grid of bench.py, ~35 s per precision), compares the oracle's two
boundary lists: length, exit flag, entering voxels, distances and segment lengths.
gpu: device name and power limit (nvidia-smi, read-only queries), then for the singlet (f64, f32) and both multiplets
(O I 102.6 nm, H Lyman; f64) on the 100x60x24x16 grid: rays per voxel in full and marched (b200rt_fold_rays), the
ray-voxel steps as the reference counts them (b200rt_last_step_count, what bench.py reports) and as executed (the steps
of the marched rays only, from the boundary lists), and the median traversal and march times of the influence build
(device events, after one warm-up build).  Writes DIR/ray_fold.json.  Needs a CUDA device: there is no fallback."""
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
BENCH_GRID = dict(shape=(100, 60, 24, 16), kw=dict(rmethod=synth.RMETHOD_ALTITUDE, rmax=synth.rMars + 50000e5))


def probe(prec, shape, chunk=64, **kw):
    from oracle import oraclebind
    oraclebind.build()
    scn = synth.make_scenario(*shape, n_em=1, **kw)
    O = oraclebind.OracleModel(scn, prec)
    nt, nph = scn.n_theta, scn.n_phi
    n_rays = nt * nph
    r = dict(grid=list(shape), prec=prec, pairs=0, length_or_flag_mismatches=0, entering_mismatches=0,
             max_rel_distance_diff=0.0, max_pair_rel_segment_diff=0.0)
    t0 = time.time()
    for v0 in range(0, scn.n_vox, chunk):
        v1 = min(scn.n_vox, v0 + chunk)
        ln, eb, ent, dist = O.traverse_voxel_rays(v0, v1)
        off = np.concatenate([[0], np.cumsum(ln)])
        for v in range(v1 - v0):
            for i in range(nt):
                for j in range(nph // 2):
                    a, b = v * n_rays + i * nph + j, v * n_rays + i * nph + (nph - 1 - j)
                    r["pairs"] += 1
                    if ln[a] != ln[b] or eb[a] != eb[b]:
                        r["length_or_flag_mismatches"] += 1
                        continue
                    if not np.array_equal(ent[off[a]:off[a + 1]], ent[off[b]:off[b + 1]]):
                        r["entering_mismatches"] += 1
                        continue
                    da, db = dist[off[a]:off[a + 1]], dist[off[b]:off[b + 1]]
                    if len(da) > 1:
                        rel = np.abs(da - db) / np.maximum(np.abs(da), 1e-300)
                        r["max_rel_distance_diff"] = max(r["max_rel_distance_diff"], float(rel.max()))
                        sa, sb = np.diff(da), np.diff(db)
                        m = (sa + sb) > 0
                        if m.any():
                            seg = np.abs(sa - sb)[m] / (sa + sb)[m]
                            r["max_pair_rel_segment_diff"] = max(r["max_pair_rel_segment_diff"], float(seg.max()))
    r["seconds"] = round(time.time() - t0, 1)
    print(json.dumps(r), flush=True)
    return r


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout
    return [dict(zip(("index", "name", "power_limit", "max_sm_clock"), (x.strip() for x in line.split(","))))
            for line in q.strip().splitlines()]


def executed_steps(ctx, g, prec, n_vox, chunk=128):
    """steps of the marched rays only: sum over voxels and representative rays of (list length - 1)"""
    rep, n_marched = binding.fold_rays(prec, g["ray_theta"], g["ray_phi"], g["ray_domega"])
    marched = rep == np.arange(len(rep))
    total = 0
    for v0 in range(0, n_vox, chunk):
        v1 = min(n_vox, v0 + chunk)
        ln = ctx.traverse_voxel_rays(v0, v1)[0].reshape(v1 - v0, len(rep))
        total += int(np.maximum(ln[:, marched] - 1, 0).sum())
    return n_marched, total


def measure(G, prec, repeats):
    g = G.g
    n_rays = len(g["ray_theta"])
    n_marched, executed = executed_steps(G.ctx, g, prec, G.scn.n_vox)
    G.build_rows()                                     # warm-up
    tr, ma, steps = [], [], 0
    for _ in range(repeats):
        _, steps = G.build_rows()
        tr.append(G.ctx.kernel_ms(binding.PH_TRAVERSE)[0])
        ma.append(G.ctx.kernel_ms(binding.PH_INFLUENCE)[0])
    return dict(rays_per_voxel=n_rays, marched_rays_per_voxel=n_marched, steps_reference_count=steps,
                steps_executed=executed, traverse_ms=float(np.median(tr)), march_ms=float(np.median(ma)),
                traverse_plus_march_ms=float(np.median(np.add(tr, ma))), note="traverse_ms includes the n_vox sun-ward "
                "rays and march_ms the single-scattering march, as bench.py's influence phases do")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("part", choices=["cpu", "gpu"])
    ap.add_argument("--big", action="store_true")
    ap.add_argument("--out")
    ap.add_argument("--repeats", type=int, default=3)
    a = ap.parse_args()
    if a.part == "cpu":
        lib = binding.load()
        for prec in (binding.F64, binding.F32):       # rays marched per voxel: a lost fold shows up here
            for n_phi in (6, 7, 12, 16, 32, 64, 128, 256, 512):
                n = 24 * n_phi
                t, p, d = np.zeros(n), np.zeros(n), np.zeros(n)
                rb = np.geomspace(3.4e8, 1.0e10, 20)
                lib.b200rt_make_grid_sph(prec, 20, 14, 24, n_phi, rb, 0, 1, np.zeros(14), np.zeros(19), np.zeros(13),
                                         t, p, d)
                print(json.dumps(dict(prec="f64" if prec == binding.F64 else "f32", n_theta=24, n_phi=n_phi, rays=n,
                                      marched=binding.fold_rays(prec, t, p, d)[1])), flush=True)
        for prec in ("f64", "f32"):
            for shape in ((12, 8, 5, 6), (20, 12, 6, 8), (40, 20, 7, 12)):
                probe(prec, shape)
            if a.big:
                probe(prec, BENCH_GRID["shape"], chunk=16, **BENCH_GRID["kw"])
        return
    if not a.out:
        ap.error("gpu needs --out DIR")
    os.makedirs(a.out, exist_ok=True)
    if binding.load().b200rt_device_count() < 1:
        raise SystemExit("no CUDA device")
    report = dict(gpus=gpu_info(), grid=list(BENCH_GRID["shape"]), builds={})
    scn = synth.make_scenario(*BENCH_GRID["shape"], n_em=1, **BENCH_GRID["kw"])
    for prec in ("f64", "f32"):
        G = binding.GpuModel(scn, prec)
        report["builds"][f"singlet_{prec}"] = r = measure(G, binding.F64 if prec == "f64" else binding.F32, a.repeats)
        print(json.dumps({f"singlet_{prec}": r}), flush=True)
        del G
    for kind, name in ((0, "O_1026"), (1, "H_lyman_multiplet")):
        M = binding.GpuMultiplet(synth.make_multiplet_scenario(kind, *BENCH_GRID["shape"], sza_T_contrast=0.1), "f64")
        report["builds"][name] = r = measure(M, binding.F64, a.repeats)
        print(json.dumps({name: r}), flush=True)
        del M
    with open(os.path.join(a.out, "ray_fold.json"), "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
