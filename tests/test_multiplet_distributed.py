"""The multiplet emissions (O I 102.6 nm, the H Lyman multiplet, the singlet through the multiplet code) in the
distributed solve: influence rows over interleaved voxel ranges, GMRES over the n_el = n_vox * n_upper element rows
(csrc/solve_krylov.cu), b200rt_solve's choice between it and the LU, and the device group.

As in test_distributed_solve.py, one GPU is enough to exercise the exchange protocol: several contexts on device 0, one
host thread each, every context holding only ITS interleaved shard of the rows."""
import importlib
import threading

import numpy as np
import pytest

from util import rel_err

pytestmark = pytest.mark.gpu

multi = importlib.import_module("3d_planetary_rt_model_b200.multi")
KINDS = [0, 1, 2]          # O_1026_emission, H_lyman_multiplet, H_lyman_singlet
SHAPE = (20, 12, 6, 8)     # 209 voxels: 627 (O I), 836 (H multiplet), 418 (singlet) elements


def dev(a, b):
    """max |a - b| / max |b|: the O I source function spans ~80 decades, so the bar is against its largest element"""
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(np.asarray(b)).max())


def run_ranks(binding, scn, devices, chunks=3, prec="f64", drop_last=False):
    """one multiplet context per entry of `devices`, each building its interleaved shard and joining the distributed
    solve (test_distributed_solve.run_ranks for GpuMultiplet)"""
    world = len(devices)
    models = [binding.GpuMultiplet(scn, prec, device=d) for d in devices]
    blocks = [m.ctx.solve_exchange()[0] for m in models]
    errors = [None] * world

    def work(r):
        try:
            ranges = multi.partition_interleaved(scn.n_vox, world, r, chunks)
            if drop_last and r == world - 1:
                ranges = ranges[:-1]
            models[r].build_ranges(ranges)
            models[r].ctx.solve_distributed(r, world, blocks)
        except Exception as ex:          # noqa: BLE001 -- reported by the caller
            errors[r] = ex

    threads = [threading.Thread(target=work, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for ex in errors:
        if ex is not None:
            raise ex
    return models


@pytest.fixture(params=["one launch", "four launches per step"])
def form(request, monkeypatch):
    """the solve as one cooperative launch (kry_loop, the default) and as the per-step launches it falls back to"""
    monkeypatch.setenv("B200RT_KRYLOV_FUSED", "1" if request.param == "one launch" else "0")
    monkeypatch.setenv("B200RT_KRYLOV_CTAS", "64")     # several ranks share device 0 here: every resident grid has to fit
    return request.param


def lu_solution(binding, scn, monkeypatch):
    monkeypatch.setenv("B200RT_SOLVER", "lu")
    G = binding.GpuMultiplet(scn, "f64")
    G.build_rows()
    G.solve()
    monkeypatch.delenv("B200RT_SOLVER")
    return G, G.vectors()["S"].copy()


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("kind", KINDS)
def test_ranges_equal_a_full_build(synth, binding, kind, prec, world):
    scn = synth.make_multiplet_scenario(kind, *SHAPE, sza_T_contrast=0.1)
    full = binding.GpuMultiplet(scn, prec)
    _, steps_full = full.build_rows()
    K = full.K()
    ref = full.vectors(want_S=False)
    nu, steps = full.n_upper, 0
    for r in range(world):
        m = binding.GpuMultiplet(scn, prec)
        _, s = m.build_ranges(multi.partition_interleaved(scn.n_vox, world, r, 3))
        steps += s
        el = [v * nu + q for a, b in multi.partition_interleaved(scn.n_vox, world, r, 3) for v in range(a, b) for q in range(nu)]
        Kr = m.K()[el]
        assert np.abs(Kr - K[el]).max() <= 1e-12 * np.abs(K).max()        # the order of the fp64 REDs
        got = m.vectors(want_S=False)
        for k in ("S0", "tau_species_ss", "tau_absorber_ss"):
            assert np.array_equal(got[k], ref[k]), k                       # every rank marches every sun-ward ray
    assert steps == steps_full


@pytest.mark.parametrize("kind", KINDS)
def test_one_rank_gmres_equals_lu(synth, binding, monkeypatch, kind, form):
    scn = synth.make_multiplet_scenario(kind, *SHAPE, sza_T_contrast=0.1)
    G, S_lu = lu_solution(binding, scn, monkeypatch)
    monkeypatch.setenv("B200RT_KRYLOV_MIN_N", "50")
    G.solve()                                                          # b200rt_solve takes the GMRES now
    launches = G.ctx.kernel_ms(binding.PH_SOLVE)[1]
    if form == "one launch":
        assert launches <= 5
    assert 3 <= G.last_solve_steps() <= 100
    assert dev(G.vectors()["S"], S_lu) < 1e-9
    assert G.ctx.residual(0) < 1e-12
    monkeypatch.setenv("B200RT_KRYLOV_MAXIT", "3")
    G.solve()                                                          # cut short -> not converged -> the LU decides
    assert G.last_solve_steps() == 3
    assert np.array_equal(G.vectors()["S"], S_lu)


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_ranks_sharing_one_device(synth, binding, monkeypatch, kind, world, form):
    scn = synth.make_multiplet_scenario(kind, *SHAPE, sza_T_contrast=0.1)
    _, S_lu = lu_solution(binding, scn, monkeypatch)
    models = run_ranks(binding, scn, [0] * world)
    ref = models[0].vectors()["S"]
    assert dev(ref, S_lu) < 1e-7
    for m in models[1:]:
        assert m.last_solve_steps() == models[0].last_solve_steps()
        assert np.array_equal(m.vectors()["S"], ref)                   # every rank ran the same arithmetic
        assert m.ctx.residual(0) == models[0].ctx.residual(0)
    assert models[0].ctx.residual(0) < 1e-12


def test_missing_shard_is_reported(synth, binding, form):
    scn = synth.make_multiplet_scenario(1, *SHAPE, sza_T_contrast=0.1)
    with pytest.raises(binding.B200RTError):
        run_ranks(binding, scn, [0, 0], drop_last=True)


def group_devices(binding, at_least=3):
    n = binding.load().b200rt_device_count()
    ids = list(range(n))
    while len(ids) < at_least:
        ids.append(0)
    return ids


def test_device_group_distributes_a_multiplet(synth, binding, monkeypatch):
    monkeypatch.setenv("B200RT_KRYLOV_MIN_N", "50")
    monkeypatch.setenv("B200RT_GROUP_MIN_LOS", "0")
    scn = synth.make_multiplet_scenario(1, *SHAPE, sza_T_contrast=0.1)
    grp = binding.GpuMultiplet(scn, "f64", devices=group_devices(binding))
    one = binding.GpuMultiplet(scn, "f64", device=0)
    one.build_rows()
    grp.ctx.generate_S()
    assert grp.ctx.residual(0) < 1e-12
    assert 3 <= grp.last_solve_steps() <= 100                          # the GMRES ran, on every member
    assert grp.ctx.kernel_ms(binding.PH_SOLVE)[1] <= 5 * grp.ctx.n_devices
    S = grp.vectors()["S"]
    monkeypatch.setenv("B200RT_SOLVER", "lu")
    one.solve()
    assert dev(S, one.vectors()["S"]) < 1e-7
    # S is resident on every member: each integrates its slice of the lines of sight with it
    one.set_sourcefn(S)
    locs, dirs = synth.random_los(301, seed=9)
    b1, bN = one.brightness(locs, dirs, 10), grp.brightness(locs, dirs, 10)
    for k in b1:
        assert np.array_equal(b1[k], bN[k]), k
    # the assembled K, gathered from the members' shards
    K1 = one.K()
    assert np.abs(grp.K() - K1).max() <= 1e-12 * np.abs(K1).max()


def test_device_group_default_grid_keeps_the_lu(synth, binding):
    """40x20 (741 voxels, below B200RT_KRYLOV_MIN_N): the rows and the LU stay on the first device, same launches"""
    scn = synth.make_multiplet_scenario(1, 40, 20, 4, 4)
    one = binding.GpuMultiplet(scn, "f64", device=0)
    grp = binding.GpuMultiplet(scn, "f64", devices=group_devices(binding))
    for m in (one, grp):
        m.build_rows()
        assert m.solve() < 1e-12
    assert grp.ctx.kernel_ms(binding.PH_SOLVE)[1] == one.ctx.kernel_ms(binding.PH_SOLVE)[1]
    assert grp.last_solve_steps() == 0
    assert rel_err(one.vectors()["S"], grp.vectors()["S"]) < 1e-10


def test_production_size_one_context(synth, binding, monkeypatch):
    """H multiplet on 100x60: n_el = 23,364 elements; a column of 99 voxels x 4 states is 4 preconditioner runs; x does
    not fit in shared memory beside a grid that owns every slice, so the one launch reads it through L2"""
    scn = synth.make_multiplet_scenario(1, 100, 60, 4, 4, sza_T_contrast=0.1)
    G = binding.GpuMultiplet(scn, "f64")
    assert G.n_el == 23364
    G.build_rows()
    G.solve()
    assert G.ctx.kernel_ms(binding.PH_SOLVE)[1] <= 5                   # the one-launch preconditioned GMRES
    steps = G.last_solve_steps()
    assert 3 <= steps <= 100
    S, res = G.vectors()["S"].copy(), G.ctx.residual(0)
    assert res < 1e-12
    monkeypatch.setenv("B200RT_SOLVER", "lu")
    G.solve()
    assert dev(S, G.vectors()["S"]) < 1e-9
