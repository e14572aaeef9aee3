"""On-disk formats, byte for byte (SURVEY.md section 8 row N3).

The reference writes its source-function and influence-matrix files with RT_grid::save_S / save_influence
(RT_grid.hpp:221-230 -> grid_spherical_azimuthally_symmetric.hpp:630-665, singlet_CFR.hpp:519-543,
emission_voxels.hpp:235-238).  oracle/_ref runs THOSE functions (the reference's own source, compiled in place); the
facade's writers (host/observation_fit.cpp write_S_file / write_influence) are given the same arrays and must produce the
same bytes.  Number formatting on the reference side is Eigen's operator<< (default IOFormat): Eigen is not vendored in
the reference tree, so oracle/standin/Eigen/Dense restates Eigen 3.4.0's print_matrix (src/Core/IO.h: every coefficient
printed at the stream's precision, all of them right-aligned to the widest) -- that one algorithm is restated, everything
else in the files is the reference's own code.  Without the reference build, test_save_S_and_influence_bytes_pins holds
the writers to the bytes of tests/golden/ref_pins.json on the oracle's arrays (pinned bit for bit to the reference's)."""
import filecmp
import importlib

import numpy as np
import pytest

import ref_pins


@pytest.fixture(scope="module")
def hb():
    return importlib.import_module("3d_planetary_rt_model_b200.host_binding")


@pytest.mark.parametrize("shape,n_em", [((8, 6, 4, 4), 2), ((12, 8, 5, 6), 1)])
def test_save_S_and_influence_bytes(synth, refbind, hb, tmp_path, shape, n_em):
    scn = synth.make_scenario(*shape, n_em=n_em, sza_T_contrast=0.1)
    R = refbind.RefModel(scn, "f64")
    R.generate_S()
    ref_S, ref_K = str(tmp_path / "ref_S.dat"), str(tmp_path / "ref_K.dat")
    R.save_S(ref_S)
    R.save_influence(ref_K)

    g = R.grid()
    names = [f"emission {e}" for e in range(n_em)]               # the names oracle/ref_harness.cpp defines
    q = np.zeros((n_em, 8, scn.n_vox))
    K = np.zeros((n_em, scn.n_vox, scn.n_vox))
    for e in range(n_em):
        a = R.arrays(e)
        v = R.vectors(e)
        sigma_ref = float(scn.em_scalars[e][2])
        q[e] = [a["density"], v["tau_species_ss"], sigma_ref * np.sqrt(a["T_ratio"]), scn.vox_in[4],
                v["tau_absorber_ss"], np.full(scn.n_vox, float(scn.abs_sigma[e])), v["S0"], v["S"]]
        K[e] = R.K(e)
    our_S, our_K = str(tmp_path / "our_S.dat"), str(tmp_path / "our_K.dat")
    hb.write_S_file(our_S, g["radial_boundaries"], g["pts_radii"], g["sza_boundaries"], g["pts_sza"], names, q)
    hb.write_influence_file(our_K, names, K)
    assert filecmp.cmp(ref_S, our_S, shallow=False), "save_S bytes differ"
    assert filecmp.cmp(ref_K, our_K, shallow=False), "save_influence bytes differ"
    txt = open(our_S).read()
    assert txt.startswith("radial boundaries [cm]: ") and "  For SZA = " in txt and "    Source function: " in txt


@pytest.mark.parametrize("shape,n_em", ref_pins.FILE_CASES)
def test_save_S_and_influence_bytes_pins(synth, oraclebind, hb, shape, n_em):
    scn = synth.make_scenario(*shape, n_em=n_em, sza_T_contrast=0.1)
    out = ref_pins.file_case(scn, oraclebind.OracleModel(scn, "f64"), hb)
    ref_pins.Pins.load().check(f"file_{'x'.join(map(str, shape))}_{n_em}", out)
