"""Line-of-sight weighting functions (b200rt_los_weights*): brightness_e = W_e S_e as a sparse matrix.

Against the device's own brightness (linearity), against the CPU oracle entry by entry (column v of W_e is the oracle's
brightness with S = e_v), the CSR structure, the products, determinism and the device group, the refusals, and the
observation_fit facade."""
import importlib
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

from util import TOL, same_bits

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STATE, ARG = 3, 2


def mixed_los(synth, scn, n, seed=11):
    """seeded lines of sight: IUVS-like ones (many hit the planet, observers inside the grid), plus observers outside
    the grid looking away from it (grid misses) and looking at the planet from outside"""
    rng = np.random.default_rng(seed)
    locs, dirs = synth.random_los(n - n // 5, seed=seed)
    k = n // 10
    rmax = scn.rb[-1]
    far = rng.normal(size=(k, 3))
    far /= np.linalg.norm(far, axis=1)[:, None]
    miss_locs = far * rmax * 1.5
    miss_dirs = far                                   # straight out: misses the grid
    m = n - len(locs) - k
    far2 = rng.normal(size=(m, 3))
    far2 /= np.linalg.norm(far2, axis=1)[:, None]
    in_locs = far2 * rmax * 1.2
    tgt = rng.normal(size=(m, 3)) * synth.rMars * 0.5
    in_dirs = tgt - in_locs
    in_dirs /= np.linalg.norm(in_dirs, axis=1)[:, None]
    return np.concatenate([locs, miss_locs, in_locs]), np.concatenate([dirs, miss_dirs, in_dirs])


def model(synth, binding, shape, prec, n_em=2, **kw):
    scn = synth.make_scenario(*shape, n_em=n_em, sza_T_contrast=0.1)
    return scn, binding.GpuModel(scn, prec, **kw)


def random_S(n_vox, e, seed=5):
    return np.random.default_rng(seed + e).uniform(0.5, 1.5, n_vox) * 1e-3 * (1 + e)


def csr(W, e, n_vox):
    indptr, indices, data = W
    return sp.csr_matrix((data[e], indices, indptr), shape=(len(indptr) - 1, n_vox))


# one emission runs lw_value_kernel<Real, 1>, two run lw_value_kernel<Real, 2> (los_weights.cu, launch_lw_values)
PREC_EM = pytest.mark.parametrize("prec,n_em", [("f64", 2), ("f32", 2), ("f64", 1), ("f32", 1)],
                                  ids=["f64", "f32", "f64-one_emission", "f32-one_emission"])


@PREC_EM
@pytest.mark.parametrize("nsub", [10, 4, 0])
@pytest.mark.parametrize("shape", [(8, 6, 4, 4), (12, 8, 5, 6), (20, 12, 6, 8)])
def test_linear_in_S_matches_device_brightness(synth, binding, shape, prec, n_em, nsub):
    scn, G = model(synth, binding, shape, prec, n_em)
    locs, dirs = mixed_los(synth, scn, 2000)
    W = G.los_weights(locs, dirs, nsub)        # before any solve or source function
    assert W[2].shape[0] == n_em
    for e in range(n_em):
        G.set_sourcefn(e, random_S(G.n_vox, e))
    _, b = G.brightness(locs, dirs, nsub)
    assert (b[:, 2] == -1).any()               # planet hits are in the set
    tol = 1e-12 if prec == "f64" else 1e-4
    for e in range(n_em):
        WS = csr(W, e, G.n_vox) @ random_S(G.n_vox, e)
        ref = b[e, 0]
        assert np.abs(ref).max() > 0
        assert np.abs(WS - ref).max() / np.abs(ref).max() < tol, (e, np.abs(WS - ref).max() / np.abs(ref).max())


@PREC_EM
def test_entries_match_oracle(synth, binding, oraclebind, prec, n_em):
    scn, G = model(synth, binding, (12, 8, 5, 6), prec, n_em)
    locs, dirs = mixed_los(synth, scn, 100, seed=3)
    indptr, indices, data = G.los_weights(locs, dirs, 10)
    O = oraclebind.OracleModel(scn, prec)
    O.build_rows()
    O.solve()
    n, nv = len(locs), G.n_vox
    dense_o = np.zeros((n_em, n, nv))
    for v in range(nv):
        ev = np.zeros(nv)
        ev[v] = 1.0
        for e in range(n_em):
            O.set_sourcefn(e, ev)
        _, bo = O.brightness(locs, dirs, 10)
        dense_o[:, :, v] = bo[:, 0]
    floor = 1e-300 if prec == "f64" else 1e-35
    stored = csr((indptr, indices, np.ones((1, len(indices)))), 0, nv).toarray() != 0
    for e in range(n_em):
        Wg = csr((indptr, indices, data), e, nv).toarray()
        Wo = dense_o[e]
        assert not (np.abs(Wo) > floor)[~stored].any(), "an oracle nonzero is not a stored entry"
        # row by row against the row's largest weight: a corner weight near 0 carries the geometry's absolute rounding
        scale = np.maximum(np.abs(Wo).max(axis=1), floor)[:, None]
        assert (np.abs(Wg - Wo) / scale).max() < TOL[prec], e


def test_structure(synth, binding):
    scn, G = model(synth, binding, (20, 12, 6, 8), "f64")
    locs, dirs = mixed_los(synth, scn, 2000)
    indptr, indices, data = G.los_weights(locs, dirs, 10)
    nnz = G.ctx.lw_nnz
    assert indptr[0] == 0 and indptr[-1] == nnz == len(indices)
    assert (np.diff(indptr) >= 0).all()
    assert ((indices >= 0) & (indices < G.n_vox)).all()
    for r in range(len(locs)):
        row = indices[indptr[r]:indptr[r + 1]]
        assert (np.diff(row) > 0).all()
    ln = G.ctx.traverse_los()[0]
    assert (ln == 0).any()
    assert (np.diff(indptr)[ln == 0] == 0).all()          # grid misses: empty rows
    assert (np.diff(indptr)[ln > 1] > 0).all()
    assert data.shape == (2, nnz) and np.isfinite(data).all()
    assert G.ctx.last_substep_count() > 0
    for ph in (binding.PH_LW_STRUCTURE, binding.PH_LW_VALUES):
        assert G.ctx.kernel_ms(ph)[1] > 0


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_products(synth, binding, prec):
    scn, G = model(synth, binding, (20, 12, 6, 8), prec)
    locs, dirs = mixed_los(synth, scn, 2000)
    W = G.los_weights(locs, dirs, 10)
    rng = np.random.default_rng(1)
    for e in range(2):
        M = csr(W, e, G.n_vox)
        x = rng.uniform(-1, 1, G.n_vox)
        r = rng.uniform(-1, 1, len(locs))
        # W x sums each row in a fixed lane order: the same bits every run, within 1e-13 of a sequential sum
        y = G.ctx.los_weights_apply(e, x)
        assert same_bits(y, G.ctx.los_weights_apply(e, x))
        assert np.abs(y - M @ x).max() <= 1e-13 * np.abs(M).dot(np.abs(x)).max()
        yt = G.ctx.los_weights_apply(e, r, transpose=True)
        assert np.abs(yt - M.T @ r).max() <= 1e-13 * np.abs(M.T).dot(np.abs(r)).max()
    assert G.ctx.kernel_ms(binding.PH_LW_APPLY)[1] == 1


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_deterministic_and_device_group(synth, binding, monkeypatch, prec):
    monkeypatch.setenv("B200RT_GROUP_MIN_LOS", "0")          # 2000 lines of sight still split over the members
    scn, G = model(synth, binding, (12, 8, 5, 6), prec)
    locs, dirs = mixed_los(synth, scn, 2000)
    a = G.los_weights(locs, dirs, 10)
    G.ctx.los_weights(10)
    b = G.ctx.los_weights_download()
    assert all(np.array_equal(p, q) for p, q in zip(a[:2], b[:2])) and same_bits(a[2], b[2])
    n = binding.load().b200rt_device_count()
    rng = np.random.default_rng(2)
    x, r = rng.uniform(0, 1, G.n_vox), rng.uniform(0, 1, len(locs))
    for ids in ([0, 0], list(range(n))):
        if len(ids) < 2:
            continue
        _, H = model(synth, binding, (12, 8, 5, 6), prec, devices=ids)
        assert H.ctx.n_devices == len(ids)
        c = H.los_weights(locs, dirs, 10)
        assert all(np.array_equal(p, q) for p, q in zip(a[:2], c[:2])) and same_bits(a[2], c[2]), ids
        for e in range(2):
            assert same_bits(G.ctx.los_weights_apply(e, x), H.ctx.los_weights_apply(e, x))
            # W^T r: members' partial vectors added on the host; the plain context adds with atomics
            yt, yh = G.ctx.los_weights_apply(e, r, True), H.ctx.los_weights_apply(e, r, True)
            assert np.abs(yt - yh).max() <= 1e-13 * np.abs(yt).max()


def status(ctx, fn, *args):
    return getattr(ctx.lib, fn)(ctx.h, *args)


def test_state_and_refusals(synth, binding):
    import ctypes as C
    scn, G = model(synth, binding, (8, 6, 4, 4), "f64")
    c = G.ctx
    nnz = C.c_longlong(0)
    assert status(c, "b200rt_los_weights", 10, C.byref(nnz)) == STATE            # no lines of sight
    locs, dirs = mixed_los(synth, scn, 200)
    c.los_upload(c.los_from_MSO(locs, dirs))
    assert status(c, "b200rt_los_weights", 1, C.byref(nnz)) == ARG
    assert status(c, "b200rt_los_weights_download", None, None, None) == STATE   # before a build
    x = np.zeros(G.n_vox)
    y = np.zeros(len(locs))
    assert status(c, "b200rt_los_weights_apply", 0, 0, x, y) == STATE
    assert c.los_weights(10) > 0                                                 # no solve, no source function
    assert status(c, "b200rt_los_weights_apply", 0, 0, x, y) == 0
    assert status(c, "b200rt_los_weights_apply", 2, 0, x, y) == ARG
    c.los_upload(c.los_from_MSO(locs[:100], dirs[:100]))                          # new lines of sight: stale
    assert status(c, "b200rt_los_weights_download", None, None, None) == STATE
    assert status(c, "b200rt_los_weights_apply", 0, 0, x, y) == STATE
    c.los_weights(0)
    c._ck(c.lib.b200rt_set_g_factor(c.h, 0, 1e-3))
    assert status(c, "b200rt_los_weights_download", None, None, None) == STATE   # new g-factor: stale

    pp = synth.make_scenario_pp(12, 4, n_em=2)
    P = binding.GpuModel(pp, "f64")
    P.ctx.los_upload(P.ctx.los_from_MSO(locs, dirs))
    assert status(P.ctx, "b200rt_los_weights", 10, C.byref(nnz)) == STATE

    M = binding.GpuMultiplet(synth.make_multiplet_scenario(0, 8, 6, 4, 4), "f64")
    M.ctx.los_upload(M.ctx.los_from_MSO(locs, dirs))
    assert status(M.ctx, "b200rt_los_weights", 10, C.byref(nnz)) == STATE


def test_facade_brightness_weights(synth):
    hb = importlib.import_module("3d_planetary_rt_model_b200.host_binding")
    F = hb.Pyobservation_fit(device=0)
    locs, dirs = synth.random_los(1500)
    F.add_observation(locs, dirs)
    F.generate_source_function(5e5, 200.0)
    b = F.brightness()
    for e in range(2):
        indptr, indices, data, shape = F.brightness_weights(e)
        assert shape == (1500, F.n_vox)
        WS = sp.csr_matrix((data, indices, indptr), shape=shape) @ F.source_function(e)
        assert np.abs(WS - b[e]).max() <= 1e-12 * np.abs(b[e]).max()
    with pytest.raises(RuntimeError):
        F.brightness_weights(0, hb.MODEL_H_PP)


def test_fast_binding_brightness_weights(synth, tmp_path):
    """the buffer-protocol .pyx path returns the facade's matrix (held to W S = brightness above)"""
    out = os.path.join(ROOT, "oracle", "_ref", "py_corona_sim_fast")
    if not (os.path.isdir(out) and any(f.startswith("py_corona_sim_gpu") and f.endswith(".so") for f in os.listdir(out))):
        pytest.skip("oracle/_ref/py_corona_sim_fast not built (needs B200RT_REFERENCE; python oracle/build_pyx.py)")
    dump = str(tmp_path / "w.npz")
    code = f"""
import importlib, sys
import numpy as np
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {out!r})
import py_corona_sim_gpu as m
synth = importlib.import_module("3d_planetary_rt_model_b200.synth")
F = m.Pyobservation_fit_b200()
locs, dirs = synth.random_los(1000)
F.add_observation(locs, dirs)
F.generate_source_function(5e5, 200.0)
np.savez({dump!r}, *[a for e in range(2) for a in F.brightness_weights(e)])
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    z = np.load(dump)
    hb = importlib.import_module("3d_planetary_rt_model_b200.host_binding")
    F = hb.Pyobservation_fit(device=0)
    locs, dirs = synth.random_los(1000)
    F.add_observation(locs, dirs)
    F.generate_source_function(5e5, 200.0)
    for e in range(2):
        indptr, indices, data, _ = F.brightness_weights(e)
        assert np.array_equal(z[f"arr_{3 * e}"], indptr) and np.array_equal(z[f"arr_{3 * e + 1}"], indices)
        assert same_bits(z[f"arr_{3 * e + 2}"], data)
