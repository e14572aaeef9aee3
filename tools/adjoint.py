"""Adjoint source-function solve (b200rt_solve_adjoint, DESIGN.md section 4) on the bench workload.

    python tools/adjoint.py --out profiles/r06_adjoint.json [--n-los 1000000] [--repeats 3]

The 100x60 grid with 24x16 rays in double, one emission (Ly alpha, bench.py's).  Alternated `repeats` times after one
warm-up of each: the forward b200rt_solve (the library's GMRES at this size: phase 2 ms and steps), the adjoint with 1 and
with 8 right-hand sides (phase 9 = the transposition of K, phase 2 = preconditioner set-up plus every iteration, steps and
true residual per right-hand side), and a device-to-device cudaMemcpyAsync of the n^2 doubles of K (torch's copy_ of
contiguous float64 tensors) to set the transposition's bytes against.  Then the O I 102.6 nm and H Lyman multiplets on
the same grid (forward and one adjoint right-hand side over n_el unknowns), and the brightness sensitivity
d(w . B)/dS0 on bench.py's seeded 10^6 lines of sight, split into the build of W (traversal, ordering, structure and value
passes), W^T w and the adjoint.  Device times from b200rt_last_kernel_ms (CUDA events); medians over the repeats.  The
card's name and power limit are read in the same run (nvidia-smi, read-only queries).  Needs a CUDA device: there is no
fallback."""
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
med = lambda v: float(np.median(v))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout
    return [dict(zip(("index", "name", "power_limit", "max_sm_clock"), (x.strip() for x in line.split(","))))
            for line in q.strip().splitlines()]


class Copy:
    """a device-to-device copy of n^2 doubles (the bytes the transposition reads and writes), device time"""

    def __init__(self, n):
        import torch
        self.torch = torch
        self.a = torch.empty(n * n, dtype=torch.float64, device="cuda:0")
        self.b = torch.empty_like(self.a)
        self.b.copy_(self.a)

    def ms(self):
        t = self.torch
        e0, e1 = t.cuda.Event(enable_timing=True), t.cuda.Event(enable_timing=True)
        e0.record()
        self.b.copy_(self.a)
        e1.record()
        t.cuda.synchronize()
        return e0.elapsed_time(e1)

    def close(self):
        del self.a, self.b
        self.torch.cuda.empty_cache()


def ph(ctx, p):
    return ctx.kernel_ms(p)[0]


def adjoint_once(ctx, e, r):
    lam, steps, res = ctx.solve_adjoint(e, r)
    return dict(transpose_ms=ph(ctx, binding.PH_TRANSPOSE), solve_ms=ph(ctx, binding.PH_SOLVE),
                launches=ctx.kernel_ms(binding.PH_SOLVE)[1], steps=steps.tolist(), residuals=res.tolist())


def summarise(runs):
    out = {k: med([r[k] for r in runs]) for k in ("transpose_ms", "solve_ms")}
    out["total_ms"] = out["transpose_ms"] + out["solve_ms"]
    out["steps"] = runs[-1]["steps"]
    out["residuals"] = runs[-1]["residuals"]
    out["launches"] = runs[-1]["launches"]
    out["runs"] = runs
    return out


def singlet(repeats, n_los):
    scn = synth.make_scenario(*GRID, n_em=1, rmethod=synth.RMETHOD_ALTITUDE, rmax=synth.rMars + 50000e5)
    G = binding.GpuModel(scn, "f64")
    c = G.ctx
    G.build_rows()
    n = G.n_vox
    rng = np.random.default_rng(7)
    r1, r8 = rng.uniform(0, 1, (1, n)), rng.uniform(0, 1, (8, n))
    copy = Copy(n)
    fwd, a1, a8, cp = [], [], [], []
    for it in range(repeats + 1):                     # the first round warms every shape up and is not kept
        c.solve()
        f = dict(ms=ph(c, binding.PH_SOLVE), steps=c.last_solve_steps(), residual=c.residual(0))
        x1, x8 = adjoint_once(c, 0, r1), adjoint_once(c, 0, r8)
        t = copy.ms()
        if it:
            fwd.append(f); a1.append(x1); a8.append(x8); cp.append(t)
    copy.close()
    kbytes = 2 * n * n * 8                            # read + written
    out = dict(n=n, forward=dict(ms=med([f["ms"] for f in fwd]), steps=fwd[-1]["steps"], residual=fwd[-1]["residual"],
                                 runs=fwd),
               adjoint_1=summarise(a1), adjoint_8=summarise(a8),
               copy_ms=med(cp), copy_ms_all=cp, copy_gbs=kbytes / (med(cp) * 1e-3) / 1e9)
    tr = med([x["transpose_ms"] for x in a1 + a8])
    out["transpose_ms"] = tr
    out["transpose_gbs"] = kbytes / (tr * 1e-3) / 1e9
    out["transpose_over_copy_bandwidth"] = med(cp) / tr
    out["adjoint_1_over_forward"] = out["adjoint_1"]["total_ms"] / out["forward"]["ms"]
    out["adjoint_steps_over_forward"] = out["adjoint_1"]["steps"][0] / out["forward"]["steps"]
    # the brightness sensitivity on bench.py's lines of sight: W, W^T w, adjoint
    locs, dirs = synth.random_los(n_los)
    w = np.random.default_rng(11).uniform(0, 1, n_los)
    c.los_upload(c.los_from_MSO(locs, dirs))
    sens = []
    for it in range(repeats + 1):
        c.los_weights(10)
        build = sum(ph(c, p) for p in (binding.PH_TRAVERSE, binding.PH_ORDER, binding.PH_LW_STRUCTURE,
                                       binding.PH_LW_VALUES))
        r = c.los_weights_apply(0, w, transpose=True)
        wt = ph(c, binding.PH_LW_APPLY)
        x = adjoint_once(c, 0, r)
        if it:
            sens.append(dict(build_W_ms=build, WT_w_ms=wt, adjoint_ms=x["transpose_ms"] + x["solve_ms"], steps=x["steps"][0],
                             residual=x["residuals"][0]))
    out["brightness_source_sensitivity"] = dict(n_los=n_los, **{k: med([s[k] for s in sens]) for k in
                                                                ("build_W_ms", "WT_w_ms", "adjoint_ms")},
                                                steps=sens[-1]["steps"], residual=sens[-1]["residual"], runs=sens)
    c.close()
    return out


def multiplet(kind, repeats):
    M = binding.GpuMultiplet(synth.make_multiplet_scenario(kind, *GRID), "f64")
    c = M.ctx
    M.build_rows()
    r = np.random.default_rng(7).uniform(0, 1, (1, M.n_el))
    fwd, adj = [], []
    for it in range(repeats + 1):
        c.solve()
        f = dict(ms=ph(c, binding.PH_SOLVE), steps=c.last_solve_steps(), residual=c.residual(0))
        x = adjoint_once(c, 0, r)
        if it:
            fwd.append(f); adj.append(x)
    out = dict(kind=["O I 102.6 nm", "H Lyman multiplet"][kind], n_el=M.n_el,
               forward=dict(ms=med([f["ms"] for f in fwd]), steps=fwd[-1]["steps"], residual=fwd[-1]["residual"]),
               adjoint_1=summarise(adj))
    out["transpose_gbs"] = 2 * M.n_el ** 2 * 8 / (out["adjoint_1"]["transpose_ms"] * 1e-3) / 1e9
    c.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n-los", type=int, default=1000000)
    ap.add_argument("--repeats", type=int, default=3)
    a = ap.parse_args()
    if binding.load().b200rt_device_count() < 1:
        raise SystemExit("no CUDA device")
    report = dict(gpus=gpu_info(), grid=list(GRID), precision="f64",
                  targets=dict(transpose_over_copy_bandwidth=">= 0.7", adjoint_steps_over_forward="within +-20 %",
                               adjoint_1_over_forward="<= 1.5 (transposition and set-up included)"))
    report["singlet"] = singlet(a.repeats, a.n_los)
    print(json.dumps({k: v for k, v in report["singlet"].items() if not isinstance(v, (dict, list))}), flush=True)
    report["multiplets"] = []
    for kind in (0, 1):
        m = multiplet(kind, a.repeats)
        print(json.dumps({k: m[k] for k in ("kind", "n_el", "forward")}), flush=True)
        report["multiplets"].append(m)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
