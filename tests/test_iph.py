"""Quemerais IPH background: oracle properties (CPU) and device parity (gpu marker).

The reference has no known-answer vector for this model and its Fortran cannot be compiled here
(parity unpinned, see oracle/iph_oracle.c); the oracle is held to the model's own invariants and the
device kernel to the oracle, at 1e-4 relative (float Real, BASELINE.json north_star)."""
import importlib
import os

import numpy as np
import pytest

from oracle import iphbind

GOLD = os.path.join(os.path.dirname(__file__), "golden", "iph_real_table.npz")
TOL = 1e-4


def golden():
    z = np.load(GOLD)
    tab = {k[4:]: z[k] for k in z.files if k.startswith("tab_")}
    for k in ("kmax", "lmax", "ninf"):
        tab[k] = int(tab[k])
    tab["temp"] = float(tab["temp"])
    return z, tab


def test_oracle_reproduces_golden_fixture():
    z, tab = golden()
    O = iphbind.IphOracle(table=tab)
    kR = O.model(float(z["g_lya"]), z["marspos"], z["ra"], z["dec"])
    assert np.array_equal(kR, z["kR"])                      # same code, same tables: bit identical
    assert 0.15 < kR.min() and kR.max() < 0.9               # ~0.2-0.8 kR across the sky from Mars' orbit


def table_file(tmp_path):
    """the reference's own table file where B200RT_REFERENCE names its tree, else the same READ sequence written from
    the committed fixture tables"""
    if iphbind.REF_TABLE and os.path.exists(iphbind.REF_TABLE):
        return iphbind.REF_TABLE
    from util import write_iph_table_file
    path = str(tmp_path / "iph_table_from_fixture")
    write_iph_table_file(golden()[1], path)
    return path


def test_written_table_file_equals_reference_file_tables(tmp_path):
    """the writer used on the GPU box reproduces, through the parser, exactly the tables of the fixture"""
    from util import write_iph_table_file
    _, tab = golden()
    path = str(tmp_path / "written")
    write_iph_table_file(tab, path)
    T = iphbind.IphOracle(fname=path).table()
    for k, v in tab.items():
        assert np.array_equal(np.asarray(v), np.asarray(T[k])), k


def test_oracle_parser_matches_fixture_tables(tmp_path):
    _, tab = golden()
    T = iphbind.IphOracle(fname=table_file(tmp_path)).table()
    for k, v in tab.items():
        assert np.array_equal(np.asarray(v), np.asarray(T[k])), k
    assert (T["kmax"], T["lmax"], T["ninf"]) == (59, 19, 5)
    assert np.allclose(T["dinf_cm3"], [0.05, 0.10, 0.15, 0.20, 0.25])
    assert T["alt_au"][0] == np.float32(0.2) and abs(T["alt_au"][-1] - 551.6) < 0.01
    assert np.array_equal(T["ang"], np.arange(19, dtype=np.float32) * 10)


def _oracle_acosf(x):
    """the acos of oracle/iph_oracle.c (and of csrc/iph.cu): a Cephes-style single-precision polynomial, restated here
    in numpy so that the two restatements can be compared on the same trajectory (see oracle/iph_numpy.py)"""
    f = np.float32

    def core(a):
        z = a * a
        p = f(4.2163199048E-2)
        for c in (2.4181311049E-2, 4.5470025998E-2, 7.4953002686E-2, 1.6666752422E-1):
            p = p * z + f(c)
        return p * z * a + a
    x = np.clip(np.asarray(x, dtype=f), f(-1), f(1))
    hi = f(2) * core(np.sqrt(f(0.5) * (f(1) - x)))
    lo = f(3.14159265358979) - f(2) * core(np.sqrt(f(0.5) * (f(1) + x)))
    mid = np.where(x >= 0, f(1.5707963267948966) - core(x), f(1.5707963267948966) + core(-x))
    return np.where(x > f(0.5), hi, np.where(x < f(-0.5), lo, mid)).astype(f)


def test_second_restatement_agrees_with_the_oracle():
    """oracle/iph_numpy.py -- written from the Fortran by a different route (vectorised numpy float32) -- against
    oracle/iph_oracle.c on the reference's own table: same outer step counts, values to 1e-5.  Catches transcription
    errors in either; the Fortran itself cannot be built here, so the row stays 'parity unpinned'."""
    import ctypes
    from oracle.iph_numpy import IphNumpy
    libm = ctypes.CDLL("libm.so.6")
    for fn in ("sinf", "cosf"):
        getattr(libm, fn).restype = ctypes.c_float
        getattr(libm, fn).argtypes = [ctypes.c_float]
    z, tab = golden()
    n = 96
    ra, dec = z["ra"][:n], z["dec"][:n]
    u = (np.cos(np.radians(dec)) * np.cos(np.radians(ra))).astype(np.float32)
    v = (np.cos(np.radians(dec)) * np.sin(np.radians(ra))).astype(np.float32)
    w = np.sin(np.radians(dec)).astype(np.float32)
    O = iphbind.IphOracle(table=tab)
    fo, so = O.background(3e11, z["marspos"], u, v, w, want_steps=True)
    N = IphNumpy(tab, sin=lambda a: libm.sinf(float(a)), cos=lambda a: libm.cosf(float(a)), acos=_oracle_acosf)
    fn_, sn = N.background(3e11, z["marspos"], u, v, w, want_steps=True)
    assert np.array_equal(so + 1, sn)          # the numpy march counts the step that leaves the model as well
    assert (np.abs(fo - fn_) / np.abs(fo)).max() < 1e-5
    # with numpy's own elementary functions the trajectories differ in the last bit, TOP's `SAB <= NORME` termination
    # flips between 20 and 21 inner steps here and there, and the two agree only to what the model itself allows
    fn2 = IphNumpy(tab).background(3e11, z["marspos"], u, v, w)
    assert (np.abs(fo - fn2) / np.abs(fo)).max() < 1e-2
    # lines of sight that pass inside the innermost node (0.2 AU): there IPAL3M returns early and the Fortran leaves FOO
    # at its previous value (:685-690 zero F and CT only) -- a corner the numpy restatement caught in iph_oracle.c and
    # the device kernel (they zeroed it; now all three follow the Fortran)
    pos = np.asarray(z["marspos"], dtype=np.float64)
    rng = np.random.default_rng(1)
    D = -pos / np.linalg.norm(pos) + 0.08 * rng.normal(size=(24, 3))
    D /= np.linalg.norm(D, axis=1)[:, None]
    assert (np.linalg.norm(np.cross(pos[None, :], D), axis=1) < 0.2).sum() >= 10
    us, vs, ws = (D[:, k].astype(np.float32) for k in range(3))
    fo3, so3 = O.background(3e11, pos, us, vs, ws, want_steps=True)
    fn3, sn3 = N.background(3e11, pos, us, vs, ws, want_steps=True)
    assert np.array_equal(so3 + 1, sn3) and (np.abs(fo3 - fn3) / np.abs(fo3)).max() < 1e-5


def test_oracle_invariants(synth):
    tab = synth.make_iph_table()
    O = iphbind.IphOracle(table=tab)
    ra, dec = synth.random_sky(300)
    g = synth.lyman_alpha_typical_g_factor
    b = O.model(g, synth.MARS_ECLIPTIC_POS, ra, dec)
    assert np.isfinite(b).all() and (b > 0).all()
    # linear in the solar flux (GRAL multiplies every term, ipbackgroundCFR_fun.f:219-221,638-647)
    b2 = O.model(2 * g, synth.MARS_ECLIPTIC_POS, ra, dec)
    assert np.allclose(b2, 2 * b, rtol=2e-6)
    # an observer beyond the last radial node sees nothing (INTENSM_PH returns at once, :598)
    far = O.model(g, (600.0, 0.0, 0.0), ra[:5], dec[:5])
    assert (far == 0).all()
    # the march takes a few hundred steps per line of sight from Mars' orbit
    u = np.cos(np.radians(dec)) * np.cos(np.radians(ra))
    v = np.cos(np.radians(dec)) * np.sin(np.radians(ra))
    w = np.sin(np.radians(dec))
    _, steps = O.background(3e11, synth.MARS_ECLIPTIC_POS, u, v, w, want_steps=True)
    assert steps.min() > 50 and steps.max() < 5000


def test_extinction_host_helper(binding):
    lib = binding.load()
    iph = np.array([1.0, 2.0, 3.0])
    tau = np.array([0.0, -1.0, 0.5])
    out = np.zeros(3)
    assert lib.b200rt_iph_extinction(3, iph, tau, out) == 0
    assert np.allclose(out, [1.0, 0.0, 3.0 * np.exp(-0.5)])      # observation.hpp:144-154


# ---------------------------------------------------------------------------------- device
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["synthetic", "real"])
def test_device_matches_oracle(synth, binding, which):
    if which == "real":
        z, tab = golden()
        ra, dec, g, pos = z["ra"], z["dec"], float(z["g_lya"]), z["marspos"]
    else:
        tab = synth.make_iph_table()
        ra, dec = synth.random_sky(4000)
        g, pos = synth.lyman_alpha_typical_g_factor, np.array(synth.MARS_ECLIPTIC_POS)
    O = iphbind.IphOracle(table=tab)
    ctx = binding.Context(0, binding.F64)
    ctx.iph_set_table(tab)
    bo = O.model(g, pos, ra, dec)
    bg = ctx.iph_model(g, pos, ra, dec)
    if which == "real":
        assert np.abs(bo - z["kR"]).max() == 0
    rel = np.abs(bo - bg) / np.abs(bo)
    assert rel.max() < TOL, rel.max()
    # the march takes the same path on both sides: identical outer step counts
    u = (np.cos(np.radians(dec)) * np.cos(np.radians(ra))).astype(np.float32)
    v = (np.cos(np.radians(dec)) * np.sin(np.radians(ra))).astype(np.float32)
    w = np.sin(np.radians(dec)).astype(np.float32)
    fo, so = O.background(3e11, pos, u, v, w, want_steps=True)
    fg, sg = ctx.iph_background(3e11, [float(x) for x in pos], u, v, w, want_steps=True)
    assert np.array_equal(so, sg)
    assert (np.abs(fo - fg) / np.abs(fo)).max() < TOL


@pytest.mark.gpu
def test_device_edge_cases(synth, binding):
    tab = synth.make_iph_table()
    ctx = binding.Context(0, binding.F64)
    with pytest.raises(binding.B200RTError):            # no table yet: state error, not garbage
        ctx.iph_model(1e-3, [1.4, 0, 0], np.array([10.0]), np.array([5.0]))
    ctx.iph_set_table(tab)
    O = iphbind.IphOracle(table=tab)
    # observer outside the model, inside the innermost node, and exactly along / against the wind axis
    for pos in ([600.0, 0.0, 0.0], [0.1, 0.05, 0.0], [1.0, 0.0, 0.0]):
        ra = np.array([0.0, 72.3, 252.3, 180.0, 359.9])
        dec = np.array([0.0, -8.7, 8.7, 89.9, -89.9])
        bo = O.model(1e-3, pos, ra, dec)
        bg = ctx.iph_model(1e-3, pos, ra, dec)
        assert np.isfinite(bg).all()
        assert np.allclose(bo, bg, rtol=TOL, atol=0)
    bad = dict(tab)
    bad["kmax"] = 100
    with pytest.raises(binding.B200RTError):
        ctx.iph_set_table(bad)


@pytest.mark.gpu
def test_device_parser(binding, tmp_path):
    _, tab = golden()
    a, b = binding.Context(0, binding.F64), binding.Context(0, binding.F64)
    a.iph_load_table(table_file(tmp_path))
    b.iph_set_table(tab)
    ra, dec = np.linspace(0, 350, 36), np.linspace(-80, 80, 36)
    assert np.array_equal(a.iph_model(2e-3, [1.41, 0.3, 0.0], ra, dec), b.iph_model(2e-3, [1.41, 0.3, 0.0], ra, dec))
