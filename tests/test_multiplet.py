"""Multiplet CFR emissions (reference emission/multiplet_CFR_emission.hpp + O_1026.hpp, H_lyman_multiplet.hpp,
H_lyman_multiplet_test.hpp; BASELINE.json configs[4] (ii)/(iii)).

CPU: the oracle restatement (oracle/multiplet_oracle.inc.c) against the reference's own source built in place
(bit for bit, double and float), against what that comparison compared against (tests/golden/ref_pins.*, for machines
without the reference build) and against golden fixtures made from it.
GPU: the CUDA path (b200rt_set_multiplet ...) against the oracle and the fixtures, 1e-6 (double) / 1e-4 (float)."""
import os

import numpy as np
import pytest

import ref_pins
from util import TOL, UNDERFLOW, rel_err, same_bits

HERE = os.path.dirname(os.path.abspath(__file__))
KINDS = [0, 1, 2]          # O_1026_emission, H_lyman_multiplet, H_lyman_singlet
GOLDEN = [(0, "f64"), (0, "f32"), (1, "f64"), (1, "f32"), (2, "f64")]


@pytest.fixture(scope="module")
def multbind():
    from oracle import multbind as mb
    return mb


def bits_equal(a, b):
    return np.array_equal(a, b) if a.dtype != np.float64 else same_bits(a, b)


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", [(8, 6, 4, 4), (12, 8, 5, 6)])
def test_oracle_matches_reference(synth, multbind, prec, kind, shape):
    if not multbind.ref_available(prec):
        pytest.skip("oracle/_ref/libref_mult_*.so not built (needs B200RT_REFERENCE)")
    scn = synth.make_multiplet_scenario(kind, *shape, sza_T_contrast=0.1)
    R, O = multbind.RefMultiplet(scn, prec), multbind.OracleMultiplet(scn, prec)
    assert (R.n_lines, R.n_mult, R.n_lower, R.n_upper, R.n_lambda) == synth.MULT_DIMS[kind]
    assert (O.n_lines, O.n_mult, O.n_lower, O.n_upper, O.n_lambda) == synth.MULT_DIMS[kind]
    cr, co = R.constants(), O.constants()
    for k in cr:
        assert bits_equal(cr[k], co[k]), k                      # constexpr tracker constants
    for line in range(R.n_lines):
        for i in range(R.n_lambda):
            for T in (131.7, 200.0, 263.1):
                assert R.lineshape(line, i, T) == O.lineshape(line, i, T)
    ar, ao = R.arrays(), O.arrays()
    for k in ar:
        assert same_bits(ar[k], ao[k]), k                       # define(): Boltzmann populations for O I
    _, ns_r = R.build_rows()
    _, ns_o = O.build_rows()
    assert ns_r == ns_o
    assert same_bits(R.K(), O.K())
    vr, vo = R.vectors(), O.vectors()
    for k in ("S0", "tau_species_ss", "tau_absorber_ss"):
        assert same_bits(vr[k], vo[k]), k
    R.solve()
    res = O.solve()
    assert res < 1e-12 if prec == "f64" else res < 1e-4
    Sr = R.vectors()["S"]
    floor = 1e-30 if prec == "f64" else float(np.abs(Sr).max())
    assert rel_err(Sr, O.vectors()["S"], floor=floor) < (1e-7 if prec == "f64" else 1e-3)
    O.set_sourcefn(Sr)
    for locs, dirs in (synth.fake_image(30 * synth.rMars, 30, 10), synth.random_los(300)):
        for nsub in (10, 0, 3):
            br, bo = R.brightness(locs, dirs, nsub), O.brightness(locs, dirs, nsub)
            for k in br:
                assert same_bits(br[k], bo[k]), (nsub, k)


def test_oracle_matches_reference_default_grid(synth, multbind):
    """reference default grid 40x20x7x12 (observation_fit.hpp:44-47), O I 102.6: a strided subset of rows"""
    if not multbind.ref_available("f64"):
        pytest.skip("oracle/_ref/libref_mult_*.so not built (needs B200RT_REFERENCE)")
    scn = synth.make_multiplet_scenario(0, 40, 20, 7, 12)
    R, O = multbind.RefMultiplet(scn), multbind.OracleMultiplet(scn)
    _, ns_r = R.build_rows(0, scn.n_vox, 97)
    _, ns_o = O.build_rows(0, scn.n_vox, 97)
    assert ns_r == ns_o
    NE, NUP = R.n_el, R.n_upper
    rows = np.concatenate([np.arange(v * NUP, (v + 1) * NUP) for v in range(0, scn.n_vox, 97)])
    assert same_bits(R.K()[rows], O.K()[rows])
    assert same_bits(R.vectors()["S0"][rows], O.vectors()["S0"][rows])


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", [(8, 6, 4, 4), (12, 8, 5, 6)])
def test_oracle_matches_reference_pins(synth, multbind, prec, kind, shape):
    pins = ref_pins.Pins.load()
    case = f"mult{kind}_{'x'.join(map(str, shape))}_{prec}"
    Sr = pins.sourcefns[case][0]
    O = multbind.OracleMultiplet(synth.make_multiplet_scenario(kind, *shape, sza_T_contrast=0.1), prec)
    out, own, res = ref_pins.mult_case(synth, O, Sr)       # brightness with the stored source function, as above
    pins.check(case, out)
    assert res < 1e-12 if prec == "f64" else res < 1e-4
    floor = 1e-30 if prec == "f64" else float(np.abs(Sr).max())
    assert rel_err(Sr, own, floor=floor) < (1e-7 if prec == "f64" else 1e-3)


def test_oracle_matches_reference_default_grid_pins(synth, multbind):
    O = multbind.OracleMultiplet(synth.make_multiplet_scenario(0, 40, 20, 7, 12))
    ref_pins.Pins.load().check("mult0_D", ref_pins.mult_grid_D_case(synth, O))


def test_singlet_through_multiplet_is_the_singlet(synth, multbind, oraclebind):
    """the reference's own consistency check (H_lyman_multiplet_test.hpp): Lyman alpha/beta through the multiplet
    code agrees with singlet_CFR to a few percent (code_todos.txt:21 reports <= 5 %; two-sided vs one-sided
    wavelength grid)"""
    scn_m = synth.make_multiplet_scenario(2, 8, 6, 4, 4)
    M = multbind.OracleMultiplet(scn_m)
    M.build_rows()
    M.solve()
    scn_s = synth.make_scenario(8, 6, 4, 4, n_em=1)
    O = oraclebind.OracleModel(scn_s)
    O.build_rows()
    O.solve()
    # single-scattering transmission: S0_singlet = T_final ; S0_multiplet(Ly a) = F n sigma / A * T_final
    c = M.constants()
    n0 = M.arrays()["species_density_0"]
    Tfin_m = M.vectors()["S0"][0::2] / (scn_m.solar[0] * n0 * c["line_sigma_total"][0] / c["upper_state_decay_rate"][0])
    Tfin_s = O.vectors(0)["S0"]
    lit = Tfin_s > 0
    assert np.abs(Tfin_m[lit] / Tfin_s[lit] - 1).max() < 0.05


def load_golden(synth, kind, prec):
    z = np.load(os.path.join(HERE, "golden", f"mult{kind}_{prec}.npz"))
    shape = tuple(int(x) for x in z["shape"])
    scn = synth.MultipletScenario(int(z["kind"]), *shape, z["rb"], float(z["rexo"]), int(z["szamethod"]),
                                  int(z["raymethod"]), z["solar"], z["vox_in"])
    return scn, z


def check_golden(M, z, prec, exact):
    tol = TOL[prec]
    c = M.constants()
    for k in c:
        assert bits_equal(c[k], z["const_" + k]) if exact or c[k].dtype != np.float64 else rel_err(c[k], z["const_" + k]) < 1e-15, k
    a = M.arrays()
    for k in a:
        assert same_bits(a[k], z["arr_" + k]) if exact else rel_err(a[k], z["arr_" + k]) < tol, k
    _, ns = M.build_rows()
    assert ns == int(z["n_steps"])
    K = M.K()
    if exact:
        assert same_bits(K, z["K"])
    else:
        floor = 1e-290 if prec == "f64" else 1e-30
        assert np.array_equal(np.abs(K) > floor, np.abs(z["K"]) > floor)
        assert rel_err(np.where(np.abs(K) > floor, K, 0), np.where(np.abs(z["K"]) > floor, z["K"], 0)) < tol
    v = M.vectors(want_S=False)
    for k in ("S0", "tau_species_ss", "tau_absorber_ss"):
        assert same_bits(v[k], z["vec_" + k]) if exact else rel_err(v[k], z["vec_" + k], floor=UNDERFLOW[prec]) < tol, k
    M.solve()
    Sg = z["vec_S"]
    floor = 1e-30 if prec == "f64" else float(np.abs(Sg).max())
    assert rel_err(M.vectors()["S"], Sg, floor=floor) < (1e-7 if prec == "f64" else 1e-3 if exact else tol)
    M.set_sourcefn(Sg)
    for nsub in (10, 0):
        b = M.brightness(z["los_loc"], z["los_dir"], nsub)
        for k in b:
            ref = z[f"b{nsub}_{k}"]
            if exact:
                assert same_bits(b[k], ref), (nsub, k)
            else:
                assert np.array_equal(b[k] == -1, ref == -1)
                assert rel_err(b[k], ref, floor=1e-300) < (tol if k == "brightness" else 2 * tol), (nsub, k)


@pytest.mark.parametrize("kind,prec", GOLDEN)
def test_oracle_reproduces_golden(synth, multbind, kind, prec):
    scn, z = load_golden(synth, kind, prec)
    check_golden(multbind.OracleMultiplet(scn, prec), z, prec, exact=True)


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("kind", KINDS)
def test_product_descriptor_equals_tracker_constants(synth, binding, multbind, kind, prec):
    """b200rt_multiplet_desc_init (host helper of the product, no GPU needed) restates the trackers' constexpr
    constants: bit-identical to the oracle's, which is pinned bit for bit to the reference build above"""
    lib = binding.load()
    d = binding.MultipletDesc()
    assert lib.b200rt_multiplet_desc_init(kind, binding.F64 if prec == "f64" else binding.F32, __import__("ctypes").byref(d)) == 0
    scn = synth.make_multiplet_scenario(kind, 8, 6, 4, 4)
    O = multbind.OracleMultiplet(scn, prec)
    c = O.constants()
    assert (d.n_lines, d.n_multiplets, d.n_lower, d.n_upper, d.n_lambda) == synth.MULT_DIMS[kind]
    NL = d.n_lines
    for name, field in (("multiplet_index", d.multiplet_index), ("lower_level_index", d.lower_level_index),
                        ("upper_level_index", d.upper_level_index)):
        assert list(field)[:NL] == list(c[name]), name
    for name, field in (("line_sigma_total", d.line_sigma_total), ("line_A", d.line_A), ("absorber_xsec", d.absorber_xsec),
                        ("offset", d.offset), ("norm", d.norm), ("weight", d.weight)):
        assert same_bits(np.array(list(field)[:NL]), c[name]), name
    assert same_bits(np.array(list(d.upper_state_decay_rate)[:d.n_upper]), c["upper_state_decay_rate"])


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_product_define_equals_reference_define(synth, binding, multbind, prec):
    """binding.define_multiplet_tables (host, numpy) against O_1026_emission::define of the oracle (Boltzmann levels)"""
    scn = synth.make_multiplet_scenario(0, 12, 8, 5, 6, sza_T_contrast=0.1)
    t = binding.define_multiplet_tables(scn, binding.F64 if prec == "f64" else binding.F32)
    a = multbind.OracleMultiplet(scn, prec).arrays()
    for l in range(3):
        assert rel_err(t["species_density"][l], a[f"species_density_{l}"]) < (1e-14 if prec == "f64" else 1e-6)
        assert rel_err(t["species_density_pt"][l], a[f"species_density_pt_{l}"]) < (1e-14 if prec == "f64" else 1e-6)


# ------------------------------------------------------------------ CUDA path
def compare_gpu(synth, O, G, prec, los_sets):
    tol = TOL[prec]
    _, ns_o = O.build_rows()
    _, ns_g = G.build_rows()
    assert ns_o == ns_g
    Ko, Kg = O.K(), G.K()
    floor = 1e-290 if prec == "f64" else 1e-30
    assert np.array_equal(np.abs(Ko) > floor, np.abs(Kg) > floor)
    assert rel_err(np.where(np.abs(Ko) > floor, Ko, 0), np.where(np.abs(Kg) > floor, Kg, 0)) < tol
    vo, vg = O.vectors(), G.vectors(want_S=False)
    for k in ("S0", "tau_species_ss", "tau_absorber_ss"):
        assert rel_err(vo[k], vg[k], floor=UNDERFLOW[prec]) < tol, k
    O.solve()
    assert G.solve() < 1e-12
    So = O.vectors()["S"]
    fl = 1e-30 if prec == "f64" else float(np.abs(So).max())
    assert rel_err(So, G.vectors()["S"], floor=fl) < tol
    G.set_sourcefn(So)
    for locs, dirs in los_sets:
        for nsub in (10, 0, 4):
            bo, bg = O.brightness(locs, dirs, nsub), G.brightness(locs, dirs, nsub)
            for k in bo:
                assert np.array_equal(bo[k] == -1, bg[k] == -1), (nsub, k)
                assert rel_err(bo[k], bg[k], floor=1e-300) < (tol if k == "brightness" else 2 * tol), (nsub, k)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", [(8, 6, 4, 4), (12, 8, 5, 6)])
def test_cuda_matches_oracle(synth, binding, multbind, prec, kind, shape):
    scn = synth.make_multiplet_scenario(kind, *shape, sza_T_contrast=0.1)
    compare_gpu(synth, multbind.OracleMultiplet(scn, prec), binding.GpuMultiplet(scn, prec), prec,
                [synth.fake_image(30 * synth.rMars, 30, 16), synth.random_los(500)])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_cuda_matches_oracle_default_grid(synth, binding, multbind, kind):
    """BASELINE.json configs[4] (ii)/(iii): O I 102.6 and the H Lyman multiplet on the reference default grid"""
    scn = synth.make_multiplet_scenario(kind, 40, 20, 7, 12)
    compare_gpu(synth, multbind.OracleMultiplet(scn), binding.GpuMultiplet(scn), "f64",
                [synth.fake_image(30 * synth.rMars, 30, 24)])


@pytest.mark.gpu
@pytest.mark.parametrize("kind,prec", GOLDEN)
def test_cuda_reproduces_golden(synth, binding, kind, prec):
    scn, z = load_golden(synth, kind, prec)
    check_golden(binding.GpuMultiplet(scn, prec), z, prec, exact=False)


@pytest.mark.gpu
def test_multiplet_then_singlet_on_one_context(synth, binding, oraclebind):
    """set_singlet after set_multiplet returns the context to singlet shapes"""
    scn_m = synth.make_multiplet_scenario(2, 8, 6, 4, 4)
    G = binding.GpuMultiplet(scn_m)
    G.build_rows()
    scn = synth.make_scenario(8, 6, 4, 4, n_em=1)
    G.ctx.set_singlet(0, 1, *(float(x) for x in scn.em_scalars[0]), binding.define_singlet_tables(scn, 0))
    G.ctx.influence()
    O = oraclebind.OracleModel(scn)
    O.build_rows()
    assert rel_err(O.K(0), G.ctx.influence_matrix(0)) < 1e-6
