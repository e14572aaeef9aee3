"""Mirror-pair fold of the voxel-origin rays (grid_host.cpp fold_pairs, b200rt_fold_rays).

Every voxel point of the azimuthally symmetric grid lies in the phi = 0 half-plane, so the rays at phi and 2 pi - phi of
one voxel cross the same voxels over the same lengths.  The influence builds march such a pair once with twice its
domega.
CPU: the premise on the oracle's boundary lists, and the fold rule through the binding.
GPU: K, S0 and the step count against the oracle on a grid that mixes folded pairs and single rays."""
import numpy as np
import pytest

from util import TOL, UNDERFLOW, rel_err

PREC = {"f64": 0, "f32": 1}


def make_rays(binding, prec, n_theta, n_phi, raymethod=1):
    lib = binding.load()
    n = n_theta * n_phi
    t, p, d = np.zeros(n), np.zeros(n), np.zeros(n)
    rb = np.geomspace(3.4e8, 1.0e10, 20)
    rc = lib.b200rt_make_grid_sph(PREC[prec], 20, 14, n_theta, n_phi, rb, 0, raymethod, np.zeros(14), np.zeros(19),
                                  np.zeros(13), t, p, d)
    assert rc == 0
    return t, p, d


# ------------------------------------------------------------------ CPU: the premise
@pytest.mark.parametrize("shape", [(12, 8, 5, 6), (20, 12, 6, 8), (40, 20, 7, 12)])
def test_mirror_rays_cross_the_same_voxels(synth, oraclebind, shape):
    """double: the reference lists of the rays phi_j and phi_(n_phi-1-j) of every voxel have the same length, flag and
    entering voxels, and distances equal to 1e-12 relative"""
    scn = synth.make_scenario(*shape, n_em=1)
    O = oraclebind.OracleModel(scn, "f64")
    nt, nph = scn.n_theta, scn.n_phi
    ln, eb, ent, dist = O.traverse_voxel_rays()
    off = np.concatenate([[0], np.cumsum(ln)])
    pairs = 0
    for v in range(scn.n_vox):
        for i in range(nt):
            for j in range(nph // 2):
                a = (v * nt + i) * nph + j
                b = (v * nt + i) * nph + nph - 1 - j
                assert ln[a] == ln[b] and eb[a] == eb[b], (v, i, j)
                assert np.array_equal(ent[off[a]:off[a + 1]], ent[off[b]:off[b + 1]]), (v, i, j)
                da, db = dist[off[a]:off[a + 1]], dist[off[b]:off[b + 1]]
                assert np.all(np.abs(da - db) <= 1e-12 * np.abs(da)), (v, i, j)
                pairs += 1
    assert pairs == scn.n_vox * nt * (nph // 2)


# ------------------------------------------------------------------ CPU: the fold rule
@pytest.mark.parametrize("n_phi", [2, 4, 6, 12, 16, 32, 64, 128, 256, 512])
@pytest.mark.parametrize("raymethod", [0, 1])
def test_even_n_phi_folds_every_mirror_pair_in_double(binding, n_phi, raymethod):
    t, p, d = make_rays(binding, "f64", 6, n_phi, raymethod)
    rep, n = binding.fold_rays(0, t, p, d)
    assert n == 6 * n_phi // 2
    for i in range(6):
        for j in range(n_phi):
            assert rep[i * n_phi + j] == i * n_phi + min(j, n_phi - 1 - j)


@pytest.mark.parametrize("n_phi", [1, 3, 7, 9])
def test_odd_n_phi_leaves_phi_pi_single(binding, n_phi):
    t, p, d = make_rays(binding, "f64", 5, n_phi)
    rep, n = binding.fold_rays(0, t, p, d)
    assert n == 5 * (n_phi + 1) // 2
    mid = n_phi // 2                                          # phi = pi
    for i in range(5):
        assert rep[i * n_phi + mid] == i * n_phi + mid
        assert np.sum(rep[i * n_phi:(i + 1) * n_phi] == i * n_phi + mid) == 1
        for j in range(n_phi):
            assert rep[i * n_phi + j] == i * n_phi + min(j, n_phi - 1 - j)


@pytest.mark.parametrize("n_phi", [6, 7, 12, 16])
def test_float_folds_only_bit_equal_rays(binding, n_phi):
    """float: phi and 2 pi - phi round to float apart, so cos(phi) of a mirror pair differs (~1e-8) and nothing folds;
    rays whose uploaded tables are bit-equal (here: the set given twice) do"""
    t, p, d = make_rays(binding, "f32", 5, n_phi)
    rep, n = binding.fold_rays(1, t, p, d)
    assert n == len(t) and np.array_equal(rep, np.arange(len(t)))
    rep2, n2 = binding.fold_rays(1, np.concatenate([t, t]), np.concatenate([p, p]), np.concatenate([d, d]))
    assert n2 == len(t)
    assert np.array_equal(rep2, np.concatenate([np.arange(len(t)), np.arange(len(t))]))


def test_asymmetric_phi_folds_nothing(binding):
    """a caller-supplied ray set whose azimuths are not mirror-symmetric, and a plane-parallel one (phi = 0)"""
    n_theta, n_phi = 5, 8
    t, _, d = make_rays(binding, "f64", n_theta, n_phi)
    p = np.tile(0.3 + np.arange(n_phi) * 2 * np.pi / n_phi, n_theta)
    for prec in (0, 1):
        rep, n = binding.fold_rays(prec, t, p, d)
        assert n == len(t) and np.array_equal(rep, np.arange(len(t)))
    tpp = np.linspace(0.1, 3.0, 7)
    rep, n = binding.fold_rays(0, tpp, np.zeros(7), np.full(7, 0.1))
    assert n == 7


def test_fold_needs_equal_domega(binding):
    t, p, d = make_rays(binding, "f64", 4, 6)
    d = d.copy()
    d[5] *= 1 + 1e-15                                         # the partner of ray 0 (theta 0, phi_5 = 2 pi - phi_0)
    rep, n = binding.fold_rays(0, t, p, d)
    assert rep[5] == 5 and n == 4 * 3 + 1


# ------------------------------------------------------------------ GPU: the folded build against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_folded_singlet_build_matches_oracle(synth, binding, oraclebind, prec):
    """20x12x6x7: odd n_phi, so every polar angle has three folded pairs (f64) and the single phi = pi ray"""
    scn = synth.make_scenario(20, 12, 6, 7, n_em=2, sza_T_contrast=0.1)
    O = oraclebind.OracleModel(scn, prec)
    G = binding.GpuModel(scn, prec)
    _, ns_o = O.build_rows()
    _, ns_g = G.build_rows()
    assert ns_o == ns_g
    tol = TOL[prec]
    floor = 1e-290 if prec == "f64" else 1e-30
    for e in range(scn.n_em):
        Ko, Kg = O.K(e), G.K(e)
        assert np.array_equal(np.abs(Ko) > floor, np.abs(Kg) > floor)
        assert rel_err(np.where(np.abs(Ko) > floor, Ko, 0), np.where(np.abs(Kg) > floor, Kg, 0)) < tol
        vo, vg = O.vectors(e), G.vectors(e, want_S=False)
        for k in ("S0", "tau_species_ss", "tau_absorber_ss"):
            assert rel_err(vo[k], vg[k], floor=UNDERFLOW[prec]) < tol, k


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_folded_multiplet_build_matches_oracle(synth, binding, prec):
    from oracle import multbind
    scn = synth.make_multiplet_scenario(0, 20, 12, 6, 7, sza_T_contrast=0.1)
    O, G = multbind.OracleMultiplet(scn, prec), binding.GpuMultiplet(scn, prec)
    _, ns_o = O.build_rows()
    _, ns_g = G.build_rows()
    assert ns_o == ns_g
    tol = TOL[prec]
    floor = 1e-290 if prec == "f64" else 1e-30
    Ko, Kg = O.K(), G.K()
    assert np.array_equal(np.abs(Ko) > floor, np.abs(Kg) > floor)
    assert rel_err(np.where(np.abs(Ko) > floor, Ko, 0), np.where(np.abs(Kg) > floor, Kg, 0)) < tol
    vo, vg = O.vectors(), G.vectors(want_S=False)
    for k in ("S0", "tau_species_ss", "tau_absorber_ss"):
        assert rel_err(vo[k], vg[k], floor=UNDERFLOW[prec]) < tol, k
