"""Pin oracle/rt_oracle.c against the reference's own source built in place (oracle/_ref).

The live comparisons run only where oracle/_ref/*.so is built; the *_pins tests hold the oracle to what those
comparisons compared against, stored in tests/golden/ref_pins.* (tests/ref_pins.py), everywhere.
"""
import numpy as np
import pytest

import ref_pins
from util import assert_lists_equal, rel_err, same_bits

SHAPES = [(8, 6, 4, 4), (12, 8, 5, 6), (20, 12, 6, 8)]


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("shape", SHAPES)
def test_oracle_matches_reference(synth, oraclebind, refbind, prec, shape):
    if not refbind.available(prec):
        pytest.skip("reference build for this precision missing")
    scn = synth.make_scenario(*shape, n_em=2, sza_T_contrast=0.1)
    R = refbind.RefModel(scn, prec)
    O = oraclebind.OracleModel(scn, prec)
    gr, go = R.grid(), O.grid()
    for k in go:
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
    tol = 1e-7 if prec == "f64" else 1e-3   # two different LUs: rounding only (componentwise, tiny S entries)
    for e in range(2):
        assert res[e] < (1e-12 if prec == "f64" else 1e-4)
        Sr = R.vectors(e)["S"]
        # f64: componentwise; f32: relative to max|S| (a float LU only resolves ~1e-7*max|S| absolutely,
        # so two float LUs already disagree by tens of percent on the smallest components)
        floor = 1e-30 if prec == "f64" else float(np.abs(Sr).max())
        assert rel_err(Sr, O.vectors(e)["S"], floor=floor) < tol
        O.set_sourcefn(e, R.vectors(e)["S"])
    for locs, dirs in (synth.fake_image(30 * synth.rMars, 30, 24), synth.random_los(600)):
        a, b = R.traverse_los(locs, dirs), O.traverse_los(locs, dirs)
        assert_lists_equal(a[:4], b[:4])
        assert same_bits(a[4], b[4])        # ray scalars r, z, t, cost, line_z, line_x
        for nsub in (10, 0, 3):
            _, br = R.brightness(locs, dirs, nsub)
            _, bo = O.brightness(locs, dirs, nsub)
            assert same_bits(br, bo), f"n_subsamples={nsub}"


def test_reference_rmethod_altitude(synth, refbind):
    """our radial-boundary generator restates get_radial_log_linear_points
    (grid/coordinate_generation.hpp:57-87): compare with the reference's own rmethod_altitude"""
    scn = synth.make_scenario(12, 8, 5, 6, n_em=1)
    R = refbind.RefModel(scn, "f64", rmethod_inject=False)
    assert same_bits(R.grid()["radial_boundaries"], scn.rb)


def test_default_grid_D(synth, oraclebind, refbind):
    """the reference default 40x20x7x12 grid (generate_source_function.cpp:95-98), 2 emissions"""
    scn = synth.make_scenario(40, 20, 7, 12, n_em=2)
    R = refbind.RefModel(scn, "f64")
    O = oraclebind.OracleModel(scn, "f64")
    assert_lists_equal(R.traverse_voxel_rays(0, 200), O.traverse_voxel_rays(0, 200))
    t = R.generate_S()     # the reference's own driver, untouched
    O.build_rows()
    O.solve()
    for e in range(2):
        assert rel_err(R.vectors(e)["S0"], O.vectors(e)["S0"]) == 0.0
        assert rel_err(R.vectors(e)["S"], O.vectors(e)["S"], floor=1e-30) < 1e-7
    assert t > 0


@pytest.fixture(scope="module")
def pins():
    return ref_pins.Pins.load()


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("shape", SHAPES)
def test_oracle_matches_reference_pins(synth, oraclebind, pins, prec, shape):
    case = f"singlet_{'x'.join(map(str, shape))}_{prec}"
    S = pins.sourcefns[case]
    O = oraclebind.OracleModel(synth.make_scenario(*shape, n_em=2, sza_T_contrast=0.1), prec)
    out, own, res = ref_pins.singlet_case(synth, O, S)      # brightness with the stored source functions, as above
    pins.check(case, out)
    for e in range(2):
        assert res[e] < (1e-12 if prec == "f64" else 1e-4)
        floor = 1e-30 if prec == "f64" else float(np.abs(S[e]).max())
        assert rel_err(S[e], own[e], floor=floor) < (1e-7 if prec == "f64" else 1e-3)


def test_reference_rmethod_altitude_pins(synth, pins):
    pins.check("rmethod_altitude", {"radial_boundaries": synth.make_scenario(12, 8, 5, 6, n_em=1).rb})


def test_default_grid_D_pins(synth, oraclebind, pins):
    out, own = ref_pins.grid_D_case(synth, oraclebind.OracleModel(synth.make_scenario(40, 20, 7, 12, n_em=2), "f64"))
    pins.check("singlet_D", out)
    for e in range(2):
        assert rel_err(pins.sourcefns["singlet_D"][e], own[e], floor=1e-30) < 1e-7
