"""Plane-parallel grid (reference grid/grid_plane_parallel.hpp; BASELINE.json configs[4] (i)):
source function only -- the reference has no interp_weights on this grid (:304-311).

CPU: the oracle restatement against the reference's own source built in place and against the
golden fixture made from it (and, without the reference build, against what the comparison with it compared against:
tests/golden/ref_pins.*).  GPU: the CUDA path (b200rt_set_grid_pp) against oracle and fixture."""
import os

import numpy as np
import pytest

import ref_pins
from util import TOL, UNDERFLOW, assert_lists_equal, rel_err, same_bits

HERE = os.path.dirname(os.path.abspath(__file__))
SHAPES = [(8, 4), (12, 5), (40, 7), (40, 6)]    # <40,7> observation_fit.hpp:48-50, <40,6> generate_source_function.cpp:85-93


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("shape", SHAPES)
def test_oracle_matches_reference_pp(synth, oraclebind, refbind, prec, shape):
    if not refbind.available(prec):
        pytest.skip("reference build for this precision missing")
    scn = synth.make_scenario_pp(*shape, n_em=2)
    R = refbind.RefModel(scn, prec)
    O = oraclebind.OracleModel(scn, prec)
    gr, go = R.grid(), O.grid()
    for k in ("pts_radii", "ray_theta", "ray_domega"):
        assert same_bits(gr[k], go[k]), k
    for e in range(2):
        ar, ao = R.arrays(e), O.arrays(e)
        for k in ar:
            assert same_bits(ar[k], ao[k]), k
    assert_lists_equal(R.traverse_voxel_rays(), O.traverse_voxel_rays())
    _, ns_r = R.build_rows()
    _, ns_o = O.build_rows()
    assert ns_r == ns_o
    for e in range(2):
        assert same_bits(R.K(e), O.K(e))
        vr, vo = R.vectors(e), O.vectors(e)
        for k in ("S0", "tau_species_ss", "tau_absorber_ss"):
            assert same_bits(vr[k], vo[k]), k
    R.solve()
    res = O.solve()
    for e in range(2):
        assert res[e] < (1e-12 if prec == "f64" else 1e-4)
        Sr = R.vectors(e)["S"]
        floor = 1e-30 if prec == "f64" else float(np.abs(Sr).max())
        assert rel_err(Sr, O.vectors(e)["S"], floor=floor) < (1e-7 if prec == "f64" else 1e-3)


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("shape", SHAPES)
def test_oracle_matches_reference_pp_pins(synth, oraclebind, prec, shape):
    pins = ref_pins.Pins.load()
    case = f"pp_{'x'.join(map(str, shape))}_{prec}"
    out, own, res = ref_pins.pp_case(oraclebind.OracleModel(synth.make_scenario_pp(*shape, n_em=2), prec))
    pins.check(case, out)
    for e in range(2):
        assert res[e] < (1e-12 if prec == "f64" else 1e-4)
        Sr = pins.sourcefns[case][e]
        floor = 1e-30 if prec == "f64" else float(np.abs(Sr).max())
        assert rel_err(Sr, own[e], floor=floor) < (1e-7 if prec == "f64" else 1e-3)


def underflow_floor(Ka, Kb, prec):
    """entries at the underflow edge of Real (against row sums of order 1) depend on the order in which the
    products of a step are formed and are compared as zeros (same rule as tests/test_gpu_parity.py)"""
    floor = 1e-290 if prec == "f64" else 1e-30
    assert np.array_equal(np.abs(Ka) > floor, np.abs(Kb) > floor)
    return np.where(np.abs(Ka) > floor, Ka, 0.0), np.where(np.abs(Kb) > floor, Kb, 0.0)


def load_pp_golden(synth, prec):
    z = np.load(os.path.join(HERE, "golden", f"pp40x7_{prec}.npz"))
    scn = synth.Scenario(40, 2, 7, 1, z["rb"], float(z["rexo"]), synth.SZAMETHOD_UNIFORM_COS, synth.RAYMETHOD_GAUSS,
                         z["em_scalars"], z["abs_sigma"], z["vox_in"], pp=True)
    return scn, z


def check_pp_golden(M, z, prec, exact):
    tol = TOL[prec]
    g = M.grid()
    for k in ("pts_radii", "ray_theta", "ray_domega"):
        assert same_bits(g[k], z["grid_" + k]), k
    assert_lists_equal(M.traverse_voxel_rays(), (z["vr_len"], z["vr_eb"], z["vr_ent"], z["vr_dist"]))
    _, nsteps = M.build_rows()
    assert nsteps == int(z["n_steps"])
    for e in range(2):
        K = M.K(e)
        if exact:
            assert same_bits(K, z[f"K{e}"])
        else:
            assert rel_err(*underflow_floor(K, z[f"K{e}"], prec)) < tol
        v = M.vectors(e, want_S=False) if not exact else M.vectors(e)
        for k in ("S0", "tau_species_ss", "tau_absorber_ss"):
            assert (same_bits(v[k], z[f"vec{e}_{k}"]) if exact else rel_err(v[k], z[f"vec{e}_{k}"], floor=UNDERFLOW[prec]) < tol), k
    M.solve()
    for e in range(2):
        Sg = z[f"vec{e}_S"]
        floor = 1e-30 if prec == "f64" else float(np.abs(Sg).max())
        assert rel_err(M.vectors(e)["S"], Sg, floor=floor) < (1e-7 if prec == "f64" else 1e-3 if exact else tol)


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_oracle_reproduces_pp_golden(synth, oraclebind, prec):
    scn, z = load_pp_golden(synth, prec)
    check_pp_golden(oraclebind.OracleModel(scn, prec), z, prec, exact=True)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_cuda_reproduces_pp_golden(synth, binding, prec):
    scn, z = load_pp_golden(synth, prec)
    check_pp_golden(binding.GpuModel(scn, prec), z, prec, exact=False)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("shape", SHAPES)
def test_cuda_matches_oracle_pp(synth, binding, oraclebind, prec, shape):
    scn = synth.make_scenario_pp(*shape, n_em=2)
    O = oraclebind.OracleModel(scn, prec)
    G = binding.GpuModel(scn, prec)
    tol = TOL[prec]
    assert_lists_equal(O.traverse_voxel_rays(), G.traverse_voxel_rays())
    _, ns_o = O.build_rows()
    _, ns_g = G.build_rows()
    assert ns_o == ns_g
    for e in range(2):
        assert rel_err(*underflow_floor(O.K(e), G.K(e), prec)) < tol
        vo, vg = O.vectors(e), G.vectors(e, want_S=False)
        for k in ("S0", "tau_species_ss", "tau_absorber_ss"):
            assert rel_err(vo[k], vg[k], floor=UNDERFLOW[prec]) < tol, k
    O.solve()
    res = G.solve()
    for e in range(2):
        assert res[e] < 1e-12
        So = O.vectors(e)["S"]
        floor = 1e-30 if prec == "f64" else float(np.abs(So).max())
        assert rel_err(So, G.vectors(e)["S"], floor=floor) < tol


@pytest.mark.gpu
def test_pp_brightness_is_a_state_error(synth, binding):
    """plane_parallel_grid::interp_weights is assert(false) in the reference (:304-311): a status here"""
    scn = synth.make_scenario_pp(8, 4, n_em=1)
    G = binding.GpuModel(scn, "f64")
    G.build_rows(); G.solve()
    locs, dirs = synth.random_los(4)
    with pytest.raises(binding.B200RTError, match="plane_parallel"):
        G.brightness(locs, dirs, 10)
