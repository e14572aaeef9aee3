#!/usr/bin/env python
"""bench.py -- the hot path of BASELINE.json on N B200s of one node.

One "step" = one complete pass of the hot path over one batch of synthetic input:
    H Ly-alpha influence matrix + single scattering on the 100x60 grid with 24x16 rays
    (5841 voxels, ~1.2e8 ray-voxel steps; BASELINE.json configs[1]),
    dense (I - K) S = S0 solve,
    brightness of --n-los (default 1e6) seeded IUVS-like lines of sight (configs[2] geometry).

value     = ray-voxel steps/s of the influence build, inputs resident in HBM, device time
            (traversal + march kernels), whole job over all ranks; los_per_s is the second half
            of the metric; job_ms is the whole step (build + exchange + solve + brightness).
e2e       = the same two numbers through the reference-facing C-ABI calls with HOST buffers
            (H2D of the tables / lines of sight and D2H of the results inside the timed region).
roofline  = the dominant kernel against the roofline that binds it.  SURVEY.md 8(d): the ray march and the brightness
            integration are FP64-INSTRUCTION bound (tables are L1/L2 resident; compulsory HBM traffic is the K write and
            the LOS in/out), so "bound" is "fp64": achieved = SURVEY's algorithmic flop-equivalents per launch / the
            kernel's measured duration, peak = the DFMA rate measured on this GPU by b200rt_measure_fp64_peaks
            (MEASURED_PEAKS.json has no FP64 entry).  The HBM view the contract asks for rides along as roofline.hbm
            (fraction tiny by construction); the solve's DMMA view is in "fp64".
cpu_baseline / --impl reference = the reference's own CPU (OpenMP) source built in place
            (oracle/_ref), on a bounded sample of the same workload.

N > 1 (torchrun): influence rows are split by source voxel; each rank DMAs its finished row batches into rank 0's
resident K over NVLink (peer memory through CUDA IPC, copy engines) while it marches the next batch; rank 0 solves and
broadcasts S (NCCL, 47 kB), lines of sight are split per GPU (no communication).
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "3d_planetary_rt_model_b200"

GRID = dict(n_rb=100, n_sb=60, n_theta=24, n_phi=16)
FLOP_EQ_PER_EMISSION_STEP = 940.0      # SURVEY.md 8(d): 20 x (exp + div + ~14 flop), phi tabulated
FLOP_EQ_PER_LOS_SUBSTEP = 1520.0       # 20 x (2 exp + div + ~14 flop) + extend/interp, per emission
FLOP_EQ_PER_QUADRATIC = 65.0           # sphere / cone intersection: ~25 flop + IEEE sqrt (~14) + 1-2 IEEE divisions (~12 each)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks and throttle reasons DURING the timed region"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.max_mhz = None

    def run(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for nme, val in zip(names, f[3:7]):
                    if val.lower().startswith("active"):
                        self.reasons.add(nme)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def make_workload(synth, n_los):
    scn = synth.make_scenario(GRID["n_rb"], GRID["n_sb"], GRID["n_theta"], GRID["n_phi"], n_em=1,
                              rmethod=synth.RMETHOD_ALTITUDE, rmax=synth.rMars + 50000e5)
    locs, dirs = synth.random_los(n_los)
    return scn, locs, dirs


def partition(n, world, rank):
    """contiguous block of source voxels / lines of sight for this rank"""
    return importlib.import_module(PKG + ".multi").partition(n, world, rank)


# --------------------------------------------------------------------------- reference arm
def run_reference(args):
    """the reference's own CPU implementation (oracle/_ref, built in place from its source) on the
    host cores of this box, on a bounded sample of the same workload"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    synth = importlib.import_module(PKG + ".synth")
    from oracle import refbind
    if not refbind.available("f64"):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libref_f64.so not built (needs B200RT_REFERENCE at build time)"}))
        return
    scn, locs, dirs = make_workload(synth, args.ref_los)
    R = refbind.RefModel(scn, "f64")
    stride = args.ref_stride
    threads = R.use_all_cores()      # torchrun exports OMP_NUM_THREADS=1: pin the OpenMP arm to every core of the box
    # source function for the brightness sample: single scattering only (no CPU solve of 5841^2)
    times_b, times_l, steps = [], [], 0
    for it in range(args.warmup + args.steps):
        tb, ns = R.build_rows(0, scn.n_vox, stride)
        if it == 0:
            R.set_sourcefn(0, R.vectors(0)["S0"])
        tl, _ = R.brightness(locs, dirs, 10)
        if it >= args.warmup:
            times_b.append(tb); times_l.append(tl); steps = ns
    tb, tl = sum(times_b), sum(times_l)
    K = len(times_b)
    v = steps * K / tb
    los = args.ref_los * K / tl
    sample = (f"every {stride}th source-voxel row of the 5841 ({steps} ray-voxel steps) and "
              f"{args.ref_los} of the lines of sight per step; S = S0 for the brightness sample")
    line = {"impl": "reference", "metric": "influence-matrix ray-voxel steps/s + observation LOS/s", "value": v,
            "unit": "ray-voxel steps/s", "los_per_s": los, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": (tb + tl) / K * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "H Ly-alpha source function on 100x60 grid, 24x16 rays + IUVS-like LOS brightness",
                       "grid": GRID, "n_emissions": 1, "n_los": args.ref_los, "sample": sample},
            "cpu_baseline": {"value": v, "unit": "ray-voxel steps/s", "los_per_s": los, "cores": threads, "kind": "reference",
                             "sample": sample},
            "e2e": {"value": v, "unit": "ray-voxel steps/s", "los_per_s": los, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# --------------------------------------------------------------------------- our arm
def cuda_array(ptr, shape, dtype="<f8"):
    class _A:
        pass
    a = _A()
    a.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": dtype, "data": (int(ptr), False), "version": 2}
    return a


DUMP_K_ROWS = 256            # rows of K written by --dump-outputs: 256 x 5841 x 8 B = 12 MB
DUMP_MAX_LOS = 1 << 20       # lines of sight written by --dump-outputs: 4 results x 2^20 x 8 B = 32 MB
DUMP_SEED = 1234


def dump_outputs(out_dir, ctx, K_t, n_vox):
    """What the last timed step computed, as a caller of that path receives it, as out_dir/<name>.npy (float64): the
    solution vectors in full, a fixed seeded sample of the rows of K and, above DUMP_MAX_LOS lines of sight, a fixed
    seeded sample of them.  The same arguments give the same inputs, so two builds can be compared file for file."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(DUMP_SEED)
    out = ctx.solution(0)                                       # S, S0, tau_species_ss, tau_absorber_ss
    rows = np.sort(rng.choice(n_vox, min(DUMP_K_ROWS, n_vox), replace=False))
    out["influence_matrix_rows"] = K_t[torch.from_numpy(rows).to(K_t.device)].cpu().numpy()
    los = ctx.los_download()                                    # brightness, optical depths, column density: (1, n_los)
    n_los = ctx.n_los
    pick = np.sort(rng.choice(n_los, DUMP_MAX_LOS, replace=False)) if n_los > DUMP_MAX_LOS else slice(None)
    out.update({k: v[0, pick] for k, v in los.items()})
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def run_ours(args):
    # stdout carries exactly one JSON line: everything a library prints there (NCCL's version banner, ...) goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the caller set it (the driver counts ranks in NCCL's INFO log); the log goes to stderr so
        # that stdout stays the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        host_group = dist.new_group(backend="gloo")   # host-only waits (rank 0's in-process arm leaves the other GPUs idle)
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")

    synth = importlib.import_module(PKG + ".synth")
    binding = importlib.import_module(PKG + ".binding")
    scn, locs, dirs = make_workload(synth, args.n_los)
    n_vox, n_los = scn.n_vox, args.n_los

    ctx = binding.Context(local, binding.F64)
    g = ctx.make_grid(scn.n_rb, scn.n_sb, scn.n_theta, scn.n_phi, scn.rb, scn.szamethod, scn.raymethod)
    ctx.set_grid(g)
    tabs = binding.define_singlet_tables(scn, 0)
    b_, T_, s_, g_ = (float(x) for x in scn.em_scalars[0])
    ctx.set_singlet(0, 1, b_, T_, s_, g_, tabs)

    multi = importlib.import_module(PKG + ".multi")
    v_ranges = multi.partition_interleaved(n_vox, world, rank)   # cost-balanced shards of source voxels
    n_rows_mine = sum(b - a for a, b in v_ranges)
    l0, l1 = partition(n_los, world, rank)
    los_all = ctx.los_from_MSO(locs, dirs)                      # host preparation (atmo_vector::ptxyz)
    # this rank's lines of sight and result buffers in page-locked host memory (what a caller streaming observations
    # would hold): the e2e arm copies from / to these inside its timed region
    los_mine = [torch.from_numpy(np.ascontiguousarray(a[l0:l1])).pin_memory().numpy() for a in los_all]
    out_pinned = [torch.empty((1, l1 - l0), dtype=torch.float64).pin_memory().numpy() for _ in range(4)]
    ctx.los_upload(los_mine)                                    # resident for the device-timed arm

    Kp, S0p, tsp, tab = ctx.influence_dev(0)
    K_t = torch.as_tensor(cuda_array(Kp, (n_vox, n_vox)), device=dev)
    S_ptr = binding.C.c_void_p()
    ctx._ck(ctx.lib.b200rt_sourcefn_dev(ctx.h, 0, binding.C.byref(S_ptr)))
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the solve: right-preconditioned GMRES over the rows where they were built (csrc/solve_krylov.cu; what the library
    # itself picks for this grid size) -- on several GPUs the ranks iterate together over peer memory: no row gather, no
    # barrier, no broadcast of S.  --solver lu: the block LU on rank 0 (rows pushed there over peer memory).
    use_gmres = args.solver in ("gmres", "auto")
    if not use_gmres:
        os.environ["B200RT_SOLVER"] = "lu"
    peer_ptrs, blocks = [], None
    if use_gmres:
        blocks = multi.connect_exchange(dist, ctx, rank, world)
    elif world > 1:
        peer_ptrs = multi.connect_row_sink(dist, ctx, rank, 0, 1)

    def gather_rows():
        """the one exchange on the path: every rank's row block -> rank 0's resident K.  The rows travel INSIDE
        ctx.influence: each finished batch is DMA'd into rank 0's K over NVLink (peer memory opened through CUDA IPC,
        copy engines) while the next batch is marched, and the call returns when this rank's rows have landed; what is
        left here is the host barrier that tells rank 0 every rank is done."""
        dist.barrier()

    def one_step():
        """-> dict of device/wall times (s) for this rank"""
        t = {}
        w0 = time.perf_counter()
        ctx.influence_ranges(v_ranges)
        t["traverse"] = ctx.kernel_ms(binding.PH_TRAVERSE)[0] * 1e-3
        t["march"] = ctx.kernel_ms(binding.PH_INFLUENCE)[0] * 1e-3
        launches = ctx.kernel_ms(binding.PH_TRAVERSE)[1] + ctx.kernel_ms(binding.PH_INFLUENCE)[1]
        t["march_launches"] = ctx.kernel_ms(binding.PH_INFLUENCE)[1] - 1      # minus the single-scattering march
        steps = ctx.last_step_count()
        w1 = time.perf_counter()
        if world > 1 and not use_gmres:                         # every rank's rows are in rank 0's K after this
            gather_rows()
        w2 = time.perf_counter()
        # row_exchange = what the exchange adds to the critical path: the un-hidden tail of the row DMA inside
        # ctx.influence (its wall time minus its kernels) + the barrier
        t["exchange"] = (w2 - w1) + max(0.0, (w1 - w0) - t["traverse"] - t["march"]) if (world > 1 and not use_gmres) else 0.0
        t["influence_tail"] = (w1 - w0) - t["traverse"] - t["march"]      # host launch/sync overhead (+ un-hidden DMA tail)
        t["barrier"] = w2 - w1
        if os.environ.get("B200RT_BENCH_DEBUG"):
            print(f"rank {rank}: influence wall {(w1 - w0) * 1e3:.3f} ms, kernels {(t['traverse'] + t['march']) * 1e3:.3f} ms, "
                  f"barrier {(w2 - w1) * 1e3:.3f} ms", file=sys.stderr, flush=True)
        if use_gmres:                                           # every rank; S is resident on every rank afterwards
            ctx.solve_distributed(rank, world, blocks)
            t["solve"] = ctx.kernel_ms(binding.PH_SOLVE)[0] * 1e-3
            t["solve_steps"] = ctx.last_solve_steps()
            launches += ctx.kernel_ms(binding.PH_SOLVE)[1]
        elif rank == 0:
            ctx.solve()
            t["solve"] = ctx.kernel_ms(binding.PH_SOLVE)[0] * 1e-3
            launches += ctx.kernel_ms(binding.PH_SOLVE)[1]
        if world > 1 and not use_gmres:
            S_t = torch.as_tensor(cuda_array(S_ptr.value, (n_vox,)), device=dev)
            dist.broadcast(S_t, src=0)
            torch.cuda.synchronize()
            if rank != 0:
                S_host = S_t.cpu().numpy()
                ctx.set_sourcefn(0, S_host)
        w3 = time.perf_counter()
        ctx.brightness_resident(10)
        t["los_traverse"] = ctx.kernel_ms(binding.PH_TRAVERSE)[0] * 1e-3
        t["brightness"] = ctx.kernel_ms(binding.PH_BRIGHTNESS)[0] * 1e-3
        t["brightness_launches"] = ctx.kernel_ms(binding.PH_BRIGHTNESS)[1]     # the march launches alone
        t["order"] = ctx.kernel_ms(binding.PH_ORDER)[0] * 1e-3                 # longest-first ordering (3 launches per batch)
        t["substeps"] = ctx.last_substep_count()
        launches += (ctx.kernel_ms(binding.PH_TRAVERSE)[1] + ctx.kernel_ms(binding.PH_BRIGHTNESS)[1] +
                     ctx.kernel_ms(binding.PH_ORDER)[1])
        ctx.synchronize()
        w4 = time.perf_counter()
        t.update(w_influence=w1 - w0, w_exchange=w2 - w1, w_solve=w3 - w2, w_brightness=w4 - w3, w_total=w4 - w0,
                 steps=steps, launches=launches)
        return t

    def e2e_step():
        """the reference-facing calls with host buffers: uploads and downloads inside the timed region"""
        w0 = time.perf_counter()
        ctx.set_singlet(0, 1, b_, T_, s_, g_, tabs)             # H2D: 8 tables
        ctx.influence_ranges(v_ranges)
        sol = ctx.solution(0, want_S=False)                     # D2H: S0 + optical depths
        w1 = time.perf_counter()
        if use_gmres and world == 1:
            ctx.solve()                                         # the reference-facing call: the library picks the GMRES itself at this size
            S = ctx.solution(0)["S"]                            # D2H: S
        elif use_gmres:
            ctx.solve_distributed(rank, world, blocks)
            S = ctx.solution(0)["S"]                            # D2H: S
        elif world > 1:
            gather_rows()
        if rank == 0 and not use_gmres:
            ctx.solve()
            S = ctx.solution(0)["S"]                            # D2H: S
        if world > 1 and not use_gmres:
            S_t = torch.as_tensor(cuda_array(S_ptr.value, (n_vox,)), device=dev)
            dist.broadcast(S_t, src=0)
            torch.cuda.synchronize()
            if rank != 0:
                ctx.set_sourcefn(0, S_t.cpu().numpy())
        w2 = time.perf_counter()
        out = ctx.brightness(los_mine, 10, out=out_pinned)      # H2D 9 arrays, kernels, D2H 4 arrays (pinned buffers)
        w3 = time.perf_counter()
        assert np.isfinite(out["brightness"]).all() and sol["S0"].max() <= 1.0
        return dict(w_influence=w1 - w0, w_solve=w2 - w1, w_brightness=w3 - w2, w_total=w3 - w0)

    # ---- device-timed arm
    sampler = ClockSampler(local) if rank == 0 else None
    recs = []
    for it in range(args.warmup + args.steps):
        flush.zero_()                                           # L2 flush between iterations (not timed)
        barrier()
        if it == args.warmup and sampler:
            sampler.start()
        rec = one_step()
        barrier()
        if it >= args.warmup:
            recs.append(rec)
    if sampler:
        sampler.stop_flag = True
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ctx, K_t, n_vox)

    def reduce_max(x):
        if world == 1:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def reduce_sum(x):
        if world == 1:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        return float(tt.item())

    K = len(recs)
    t_infl = reduce_max(sum(r["traverse"] + r["march"] for r in recs))            # device time, max over ranks
    t_bright = reduce_max(sum(r["los_traverse"] + r["order"] + r["brightness"] for r in recs))
    t_solve = reduce_max(sum(r.get("solve", 0.0) for r in recs))
    t_total = reduce_max(sum(r["w_total"] for r in recs))
    t_exch = reduce_max(sum(r["exchange"] for r in recs))
    steps_total = reduce_sum(float(recs[-1]["steps"]))
    launches = int(reduce_sum(float(sum(r["launches"] for r in recs))))
    value = steps_total * K / t_infl
    los_per_s = n_los * K / t_bright

    # ---- e2e arm (host buffers)
    erecs = []
    for it in range(args.warmup + args.steps):
        flush.zero_()
        barrier()
        r = e2e_step()
        barrier()
        if it >= args.warmup:
            erecs.append(r)
    Ke = len(erecs)
    e_infl = reduce_max(sum(r["w_influence"] for r in erecs))
    e_bright = reduce_max(sum(r["w_brightness"] for r in erecs))
    e_total = reduce_max(sum(r["w_total"] for r in erecs))
    h2d = 8 * n_vox * 8 + 9 * (l1 - l0) * 8
    d2h = 4 * n_vox * 8 + 4 * (l1 - l0) * 8

    if world > 1:                     # peers let go of rank 0's K / of each other's exchange blocks before they are freed
        for p_ in peer_ptrs:
            ctx.ipc_close(p_)
        if blocks:
            for q, p_ in enumerate(blocks):
                if q != rank:
                    ctx.ipc_close(p_)
        dist.barrier()
    dfma = dmma = None
    if rank == 0:
        dfma, dmma = ctx.fp64_peaks()
    final_S = ctx.solution(0)["S"] if rank == 0 else None
    # every rank frees its GPU before rank 0 drives all of them from one process
    ctx.close()
    del flush, K_t
    torch.cuda.empty_cache()
    if rank != 0:
        dist.barrier(group=host_group)          # host-side wait: no kernel spins on this GPU meanwhile
        dist.destroy_process_group()
        return

    # ---- rooflines (device times from CUDA events on the ctx stream; SURVEY.md 8(d) algorithmic work per unit)
    hbm_peak, peak_kind = load_peaks()
    fp64_peak = max(dfma, dmma)     # the FP64 pipe: the DFMA probe reads ~10 % below the DMMA probe on the same pipe
    K = len(recs)
    mean = lambda k: sum(r[k] for r in recs) / K
    traffic = {}
    tj = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tj):
        traffic = json.load(open(tj))
    steps_rank, substeps_rank = recs[-1]["steps"], recs[-1]["substeps"]
    n_rays_rank = n_rows_mine * scn.n_rays + n_vox                   # voxel-origin rays + the sun-ward rays
    quad = GRID["n_rb"] + GRID["n_sb"] - 2                           # primitives a ray is tested against

    def roof(kernel, seconds, flop, alg_bytes, units, key, launches=1):
        dur = seconds / max(1, launches)
        return {"kernel": kernel, "bound": "fp64", "achieved": flop / seconds / 1e12, "peak": fp64_peak, "unit": "TFLOP/s",
                "frac": flop / seconds / 1e12 / fp64_peak, "peak_kind": "FP64 pipe, measured in this run (max of the DFMA and DMMA probes)",
                "frac_of_dfma_probe": flop / seconds / 1e12 / dfma, "units_per_launch": units, "launch_ms": dur * 1e3,
                "traffic": traffic.get(key),
                "hbm": {"achieved": alg_bytes / seconds / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": alg_bytes / seconds / 1e9 / hbm_peak, "peak_kind": peak_kind}}

    rooflines = {
        "brightness": roof("brightness_kernel<double,1>", mean("brightness"), substeps_rank * FLOP_EQ_PER_LOS_SUBSTEP,
                           (l1 - l0) * (6 * 8 + 4 * 8), {"los_substeps": substeps_rank, "flop_eq_per_substep": FLOP_EQ_PER_LOS_SUBSTEP},
                           "brightness_kernel", recs[-1]["brightness_launches"]),
        "march": roof("march_kernel<double,0>", mean("march"), steps_rank * FLOP_EQ_PER_EMISSION_STEP, n_rows_mine * n_vox * 8,
                      {"ray_voxel_steps": steps_rank, "flop_eq_per_step": FLOP_EQ_PER_EMISSION_STEP}, "march_kernel",
                      max(1, recs[-1]["march_launches"])),
        # traversal: (n_rb + n_sb - 2) quadratics per ray, each ~25 flop + an IEEE sqrt (~14 FP64 instructions) and one or
        # two IEEE divisions (~12 each): FLOP_EQ_PER_QUADRATIC; the ordering / merge is integer work on top
        "traverse_voxel_rays": roof("traverse_fast_kernel<double,voxel rays>", mean("traverse"),
                                    n_rays_rank * quad * FLOP_EQ_PER_QUADRATIC, steps_rank * 12.0,
                                    {"rays": n_rays_rank, "quadratics_per_ray": quad, "flop_eq_per_quadratic": FLOP_EQ_PER_QUADRATIC},
                                    "traverse_kernel"),
        "traverse_los": roof("traverse_fast_kernel<double,lines of sight>", mean("los_traverse"),
                             (l1 - l0) * quad * FLOP_EQ_PER_QUADRATIC, substeps_rank / 9.0 * 12.0,
                             {"rays": l1 - l0, "quadratics_per_ray": quad, "flop_eq_per_quadratic": FLOP_EQ_PER_QUADRATIC}, "traverse_los"),
    }
    if t_solve > 0 and use_gmres:
        sv = t_solve / K
        products = recs[-1]["solve_steps"] + 1                       # Arnoldi steps + the residual check
        k_bytes = (products + 4) * n_rows_mine * n_vox * 8.0         # + the set-up: rows read and written twice
        rooflines["solve"] = {"kernel": "distributed GMRES (kry_post: this rank's rows of K x vector, once per step)", "bound": "hbm",
                              "achieved": k_bytes / sv / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": k_bytes / sv / 1e9 / hbm_peak,
                              "peak_kind": peak_kind, "launch_ms": sv * 1e3, "steps": recs[-1]["solve_steps"],
                              "traffic": traffic.get("kry_loop"),
                              "note": "algorithmic bytes = (steps + 1 + 4) x own rows x n_vox x 8 (one product per step, the "
                                      "residual check, the preconditioner set-up's two passes over the rows); the rest of a "
                                      "step is the orthogonalisation (~13 us) and the wait for the peers' pieces"}
    elif t_solve > 0:
        sv = t_solve / K
        rooflines["solve"] = {"kernel": "block LU (gemm128 DMMA.8x8x4 + cluster Gauss-Jordan)", "bound": "fp64 tensor",
                              "achieved": (2.0 / 3.0 * n_vox ** 3) / sv / 1e12, "peak": dmma, "unit": "TFLOP/s",
                              "frac": (2.0 / 3.0 * n_vox ** 3) / sv / 1e12 / dmma, "peak_kind": "DMMA.8x8x4, measured in this run",
                              "launch_ms": sv * 1e3, "traffic": traffic.get("gemm128_kernel")}
    dominant = max(("brightness", "march", "traverse_voxel_rays", "traverse_los"), key=lambda k: rooflines[k]["launch_ms"])
    roofl = dict(rooflines[dominant])
    roofl["note"] = ("FP64-instruction bound kernels (SURVEY.md 8(d)): achieved = algorithmic flop-equivalents / measured time; "
                     "ncu's executed-instruction view of the same kernel (FP64 pipe active) is in profiles/ and is lower "
                     "(brightness 0.65): the flop-equivalent count prices exp and division at the library's instruction "
                     "counts.  roofline.hbm is small by construction")
    fp64 = {"dfma_peak_tflops": dfma, "dmma_peak_tflops": dmma,
            "march_flop_eq_tflops": rooflines["march"]["achieved"], "brightness_flop_eq_tflops": rooflines["brightness"]["achieved"],
            "los_substeps": substeps_rank,
            "solve_tflops": None if use_gmres else rooflines.get("solve", {}).get("achieved"),
            "solve_frac_of_dmma": None if use_gmres else rooflines.get("solve", {}).get("frac")}

    line = {"metric": "influence-matrix ray-voxel steps/s + observation LOS/s", "value": value,
            "unit": "ray-voxel steps/s", "los_per_s": los_per_s, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_total / K * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "H Ly-alpha source function on 100x60 grid, 24x16 rays (5841 voxels) + "
                                   f"{n_los} IUVS-like LOS brightness, n_subsamples=10",
                       "grid": GRID, "n_emissions": 1, "n_los": n_los, "ray_voxel_steps": int(steps_total),
                       "l2": "256 MB buffer written between timed iterations (L2 flush); K is 273 MB > L2",
                       "solver": ("GMRES over the ranks' resident rows (b200rt_solve_distributed), right-preconditioned with the "
                                  "inverted diagonal blocks of the SZA columns, tolerance 1e-13, "
                                  f"{recs[-1].get('solve_steps')} steps") if use_gmres else "block LU (DMMA) on one GPU",
                       "partition": ("one process per GPU: rows by source voxel, " +
                                     ("left where they were built (the ranks solve together over peer memory: no row gather, "
                                      "no host barrier, no broadcast of S)" if use_gmres else
                                      "pushed to rank 0 over peer memory while marching") +
                                     ", LOS by index; the in-process form of the same partition (one handle, "
                                     "b200rt_create_multi, what observation_fit uses) is timed under in_process")
                       if world > 1 else "single GPU"},
            "phases_ms": {"influence_traverse+march": t_infl / K * 1e3, "influence_traverse": mean("traverse") * 1e3,
                          "influence_march": mean("march") * 1e3, "row_exchange": t_exch / K * 1e3,
                          "solve": t_solve / K * 1e3, "brightness_traverse+march": t_bright / K * 1e3,
                          "los_traverse": mean("los_traverse") * 1e3, "los_order": mean("order") * 1e3,
                          "brightness_march": mean("brightness") * 1e3, "note": "rank 0 where per-kernel"},
            "exchange_detail_ms": {"influence_call_minus_kernels": sum(r["influence_tail"] for r in recs) / K * 1e3,
                                   "barrier": sum(r["barrier"] for r in recs) / K * 1e3, "note": "rank 0"},
            "solve_gflops": fp64["solve_tflops"] * 1e3 if fp64["solve_tflops"] else None,
            "roofline": roofl, "rooflines": rooflines, "fp64": fp64,
            "e2e": {"value": steps_total * Ke / e_infl, "unit": "ray-voxel steps/s", "los_per_s": n_los * Ke / e_bright,
                    "job_ms": e_total / Ke * 1e3, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": launches,
            "clocks": sampler.summary() if sampler else None}

    # ---- the same job through ONE handle in ONE process (b200rt_create_multi: what observation_fit and the RT_grid
    # binding use): rank 0 drives all N GPUs, host buffers in and out; the other ranks' GPUs are free by now
    if world > 1 and not args.no_in_process:
        try:
            line["in_process"] = run_in_process(binding, torch, scn, tabs, (b_, T_, s_, g_), los_all, world, args.warmup, args.steps)
        except Exception as ex:
            line["in_process"] = {"error": str(ex)}

    # ---- CPU baseline beside it (rank 0, N = 1 only): the reference's own source, bounded sample
    if world == 1 and not args.no_cpu_baseline:
        try:
            from oracle import refbind
            if refbind.available("f64"):
                R = refbind.RefModel(scn, "f64")
                cores = R.use_all_cores()
                tb, ns = R.build_rows(0, n_vox, args.ref_stride)
                R.set_sourcefn(0, final_S)
                tl, _ = R.brightness(locs[:args.ref_los], dirs[:args.ref_los], 10)
                line["cpu_baseline"] = {"value": ns / tb, "unit": "ray-voxel steps/s", "los_per_s": args.ref_los / tl,
                                        "cores": cores, "kind": "reference",
                                        "sample": f"every {args.ref_stride}th source-voxel row ({ns} steps, {tb:.1f} s) and "
                                                  f"{args.ref_los} lines of sight ({tl:.1f} s)"}
            else:
                from oracle import oraclebind
                O = oraclebind.OracleModel(scn, "f64")
                tb, ns = O.build_rows(0, n_vox, args.ref_stride)
                O.set_sourcefn(0, final_S)
                tl, _ = O.brightness(locs[:args.ref_los], dirs[:args.ref_los], 10)
                line["cpu_baseline"] = {"value": ns / tb, "unit": "ray-voxel steps/s", "los_per_s": args.ref_los / tl,
                                        "cores": os.cpu_count(), "kind": "port",
                                        "sample": f"every {args.ref_stride}th source-voxel row ({ns} steps) and {args.ref_los} LOS"}
        except Exception as ex:   # the baseline is a reported number, never a reason to lose the bench line
            line["cpu_baseline"] = {"error": str(ex)}
    # ---- the other configs of BASELINE.json that are not part of the timed step: the Quemerais IPH background for the
    # same lines of sight (real table, LOS split over the GPUs) and the 512-set (nH, T) sweep on grid D (sets over the
    # GPUs); at N = 1 also the multiplet emissions and the float build of the job
    if not args.no_extras:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import extra_bench
            ex = extra_bench.iph(n_los, world)
            # worker threads = contexts x GPUs.  Measured on an 8-GPU box (tools/dev/sweep_gpus.py): 8 GPUs x 1 / 2 / 3 / 4
            # contexts 1747 / 1823 / 1520 / 1230 sets/s, 4 GPUs 1185 / 1660 / 1668 / 1594, 1 GPU best at 4: beyond ~16
            # threads the process-wide host side of the runtime, not the GPUs, sets the rate
            ex.update(extra_bench.sweep(512, 10000, 4 if world <= 2 else 2, world))
            if world == 1:
                ex.update(extra_bench.multiplet(0))
                ex.update(extra_bench.multiplet(1))
                ex.update(extra_bench.float_job(n_los))
            line["extras"] = ex
        except Exception as exn:
            line["extras"] = {"error": str(exn)}
    emit(line)
    if world > 1:
        dist.barrier(group=host_group)
        dist.destroy_process_group()


def run_in_process(binding, torch, scn, tabs, scalars, los_all, n_dev, warmup, reps):
    """source function + brightness through ONE handle over n_dev GPUs of this process, host buffers in and out"""
    b_, T_, s_, g_ = scalars
    ctx = binding.Context(precision=binding.F64, devices=list(range(n_dev)))
    g = ctx.make_grid(scn.n_rb, scn.n_sb, scn.n_theta, scn.n_phi, scn.rb, scn.szamethod, scn.raymethod)
    ctx.set_grid(g)
    n_los = len(los_all[0])
    los_pin = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy() for a in los_all]
    out_pin = [torch.empty((1, n_los), dtype=torch.float64).pin_memory().numpy() for _ in range(4)]
    rec = []
    for it in range(warmup + reps):
        w0 = time.perf_counter()
        ctx.set_singlet(0, 1, b_, T_, s_, g_, tabs)             # H2D: 8 tables, every device
        ctx.generate_S()                                        # rows on every device -> device 0's K, solve, S to all
        sol = ctx.solution(0)                                   # D2H: S, S0, optical depths
        w1 = time.perf_counter()
        ph = {k: ctx.kernel_ms(p)[0] for k, p in (("traverse", binding.PH_TRAVERSE), ("march", binding.PH_INFLUENCE),
                                                   ("solve", binding.PH_SOLVE))}
        steps = ctx.last_step_count()
        out = ctx.brightness(los_pin, 10, out=out_pin)          # H2D 9 arrays / kernels / D2H 4 arrays, per device slice
        w2 = time.perf_counter()
        ph.update({k: ctx.kernel_ms(p)[0] for k, p in (("los_traverse", binding.PH_TRAVERSE), ("brightness", binding.PH_BRIGHTNESS))})
        assert np.isfinite(out["brightness"]).all() and sol["S0"].max() <= 1.0
        if it >= warmup:
            rec.append(dict(source_function_ms=(w1 - w0) * 1e3, brightness_ms=(w2 - w1) * 1e3, job_ms=(w2 - w0) * 1e3, steps=steps, **ph))
    ctx.close()
    m = lambda k: sum(r[k] for r in rec) / len(rec)
    return {"n_devices": n_dev, "job_ms": m("job_ms"), "source_function_ms": m("source_function_ms"), "brightness_ms": m("brightness_ms"),
            "value": rec[-1]["steps"] / (m("source_function_ms") * 1e-3), "unit": "ray-voxel steps/s (source function wall time incl. solve and copies)",
            "los_per_s": n_los / (m("brightness_ms") * 1e-3),
            "kernel_ms_slowest_device": {k: m(k) for k in ("traverse", "march", "solve", "los_traverse", "brightness")},
            "partition": "in-process: one handle (b200rt_create_multi), rows by source voxel into device 0's K over peer "
                         "memory, solve on device 0, S to all, LOS by index; host buffers in and out"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n-los", type=int, default=1000000)
    ap.add_argument("--ref-stride", type=int, default=8, help="CPU sample: every k-th source-voxel row")
    ap.add_argument("--ref-los", type=int, default=50000, help="CPU sample: lines of sight per step")
    ap.add_argument("--solver", default="auto", choices=["auto", "lu", "gmres"],
                    help="auto / gmres: preconditioned GMRES over the rows where they were built; lu: block LU on rank 0")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the IPH and sweep measurements")
    ap.add_argument("--no-in-process", action="store_true", help="N > 1: skip the one-handle in-process arm on rank 0")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (one process only)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        ap.error("--dump-outputs writes the results of one process; run it without torchrun")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
