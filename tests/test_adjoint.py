"""Adjoint source-function solve (b200rt_solve_adjoint): lambda = (I - w K)^-T r on the resident influence matrix.

Against the dense numpy solve of the transposed system, the identities r . S = lambda . S0 and
sum_l w_l B_l = lambda . S0 (lambda = adjoint(W^T w)) on device quantities, the solver's forms, determinism, the
forward state left untouched (plain context and a device group with distributed rows), the device group against a plain
context, the refusals, and the observation_fit facade."""
import ctypes as C
import importlib
import os
import subprocess
import sys

import numpy as np
import pytest

from test_los_weights import mixed_los
from util import rel_err, same_bits

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARG, STATE, NOT_DOMINANT = 2, 3, 5
BIG = (50, 50, 4, 4)                  # 2401 voxels: above B200RT_KRYLOV_MIN_N


def model(synth, binding, shape, prec="f64", **kw):
    scn = synth.make_scenario(*shape, n_em=2, sza_T_contrast=0.1)
    return scn, binding.GpuModel(scn, prec, **kw)


def branching(scn, e):
    return float(scn.em_scalars[e][0])


def dense_adjoint(K, w, r):
    return np.linalg.solve((np.eye(len(K)) - w * K).T, r.T).T


def check_dense(lam, res, ref):
    assert np.abs(lam - ref).max() <= 1e-10 * np.abs(ref).max()
    assert (np.asarray(res) <= 1e-8).all()


def rhs(n, k, seed=7):
    return np.random.default_rng(seed).uniform(-1.0, 1.0, (k, n))


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("shape", [(12, 8, 5, 6), (20, 12, 6, 8), BIG])
def test_matches_dense_solve(synth, binding, shape, prec):
    scn, G = model(synth, binding, shape, prec)
    G.build_rows()
    assert {round(branching(scn, e), 4) for e in range(2)} == {1.0, 0.8819}
    for e in range(2):
        K = G.K(e)
        for k in (1, 3):
            r = rhs(G.n_vox, k, seed=e + k)
            lam, steps, res = G.solve_adjoint(e, r)
            check_dense(lam, res, dense_adjoint(K, branching(scn, e), r))
            assert (steps > 0).all()
        lam1, _, _ = G.solve_adjoint(e, r[0])                # a 1-D right-hand side
        assert lam1.shape == (G.n_vox,)
    assert G.ctx.kernel_ms(binding.PH_TRANSPOSE)[1] == 1
    assert G.ctx.kernel_ms(binding.PH_SOLVE)[1] >= 1


@pytest.mark.parametrize("kind", [0, 1])
def test_multiplet_matches_dense_solve(synth, binding, kind):
    M = binding.GpuMultiplet(synth.make_multiplet_scenario(kind, 8, 6, 4, 4), "f64")
    M.build_rows()
    K = M.K()
    r = rhs(M.n_el, 3)
    lam, steps, res = M.solve_adjoint(r)
    check_dense(lam, res, dense_adjoint(K, 1.0, r))
    M.solve()
    v = M.vectors()
    assert abs(r[0] @ v["S"] - lam[0] @ v["S0"]) <= 1e-10 * abs(r[0] @ v["S"])


@pytest.mark.parametrize("solver", ["lu", "gmres"])
def test_identity_r_S(synth, binding, monkeypatch, solver):
    monkeypatch.setenv("B200RT_SOLVER", solver)
    scn, G = model(synth, binding, (20, 12, 6, 8))
    G.build_rows()
    G.solve()
    assert (G.ctx.last_solve_steps() > 0) == (solver == "gmres")
    r = rhs(G.n_vox, 2)
    for e in range(2):
        v = G.vectors(e)
        lam, _, _ = G.solve_adjoint(e, r)
        for k in range(2):
            rs = r[k] @ v["S"]
            assert abs(rs - lam[k] @ v["S0"]) <= 1e-10 * np.abs(r[k]).dot(np.abs(v["S"]))


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_identity_brightness(synth, binding, prec):
    scn, G = model(synth, binding, (20, 12, 6, 8), prec)
    G.build_rows()
    G.solve()
    locs, dirs = mixed_los(synth, scn, 2000)
    w = np.random.default_rng(3).uniform(0.0, 1.0, len(locs))
    _, b = G.brightness(locs, dirs, 10)
    for e in range(2):
        lam = G.brightness_source_sensitivity(locs, dirs, w, e)
        lhs = w @ b[e, 0]
        assert lhs > 0
        assert abs(lhs - lam @ G.vectors(e)["S0"]) <= (1e-11 if prec == "f64" else 1e-4) * lhs


@pytest.mark.parametrize("form", ["pc0", "fused0", "pp"])
def test_forms(synth, binding, monkeypatch, form):
    if form == "pc0":
        monkeypatch.setenv("B200RT_KRYLOV_PC", "0")
    if form == "fused0":
        monkeypatch.setenv("B200RT_KRYLOV_FUSED", "0")               # the per-step launches
    if form == "pp":
        scn = synth.make_scenario_pp(40, 7, n_em=2)
        G = binding.GpuModel(scn, "f64")
    else:
        scn, G = model(synth, binding, (20, 12, 6, 8))
    G.build_rows()
    r = rhs(G.n_vox, 2)
    for e in range(2):
        lam, steps, res = G.solve_adjoint(e, r)
        check_dense(lam, res, dense_adjoint(G.K(e), branching(scn, e), r))
    if form == "fused0":
        assert G.ctx.kernel_ms(binding.PH_SOLVE)[1] > 10


def test_deterministic(synth, binding):
    scn, G = model(synth, binding, (20, 12, 6, 8))
    G.build_rows()
    r = rhs(G.n_vox, 3)
    a, sa, ra = G.solve_adjoint(0, r)
    b, sb, rb = G.solve_adjoint(0, r)
    assert same_bits(a, b) and np.array_equal(sa, sb) and same_bits(ra, rb)
    for k in range(3):
        c, sc, rc = G.solve_adjoint(0, r[k])
        assert same_bits(a[k], c) and sa[k] == sc[0] and same_bits(ra[k], rc)


def forward_state(G, locs, dirs):
    return ([G.vectors(e)["S"] for e in range(2)], [G.ctx.residual(e) for e in range(2)], G.ctx.last_solve_steps(),
            G.brightness(locs, dirs, 10)[1])


def same_state(p, q):
    return (all(same_bits(a, b) for a, b in zip(p[0], q[0])) and same_bits(p[1], q[1]) and p[2] == q[2]
            and same_bits(p[3], q[3]))


def test_forward_state_untouched(synth, binding, monkeypatch):
    monkeypatch.setenv("B200RT_SOLVER", "gmres")
    scn, G = model(synth, binding, (20, 12, 6, 8))
    G.build_rows()
    G.solve()
    locs, dirs = synth.random_los(500, seed=4)
    before = forward_state(G, locs, dirs)
    G.solve_adjoint(1, rhs(G.n_vox, 2))
    assert same_state(before, forward_state(G, locs, dirs))
    G.solve()                                                   # a forward solve after the adjoint
    assert same_state(before, forward_state(G, locs, dirs))


def test_device_group_distributed_rows(synth, binding, monkeypatch):
    """device 0 named twice, rows left on the members: forward, adjoint, forward.  The adjoint must not advance the
    exchange blocks' round counters the members agree on"""
    monkeypatch.setenv("B200RT_GROUP_MIN_RAYS", "0")
    scn, H = model(synth, binding, BIG, devices=[0, 0])
    H.ctx.generate_S()
    steps = H.ctx.last_solve_steps()
    assert steps > 0
    S = [H.vectors(e)["S"] for e in range(2)]
    r = rhs(H.n_vox, 2)
    lam_g = [H.solve_adjoint(e, r)[0] for e in range(2)]
    H.ctx.solve()
    assert H.ctx.last_solve_steps() == steps
    assert all(same_bits(S[e], H.vectors(e)["S"]) for e in range(2))
    _, G = model(synth, binding, BIG)
    G.build_rows()
    for e in range(2):
        lam, _, _ = G.solve_adjoint(e, r)
        assert rel_err(lam, lam_g[e]) < 1e-12                     # K differs by the rounding of the RED order


def test_device_group_lu_form(synth, binding, monkeypatch):
    """a small grid: emission e's rows are gathered on member e (owners differ)"""
    monkeypatch.setenv("B200RT_GROUP_MIN_RAYS", "0")
    scn, H = model(synth, binding, (12, 8, 5, 6), devices=[0, 0])
    H.ctx.generate_S()
    _, G = model(synth, binding, (12, 8, 5, 6))
    G.build_rows()
    r = rhs(G.n_vox, 2)
    for e in range(2):
        assert rel_err(G.solve_adjoint(e, r)[0], H.solve_adjoint(e, r)[0]) < 1e-12


def adjoint_status(ctx, e, n_rhs, r, lam):
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    return ctx.lib.b200rt_solve_adjoint(ctx.h, e, n_rhs, p(r), p(lam), None, None)


def test_refusals(synth, binding, monkeypatch):
    scn, G = model(synth, binding, (12, 8, 5, 6))
    c, n = G.ctx, G.n_vox
    r, lam = rhs(n, 1), np.zeros((1, n))
    assert adjoint_status(c, 0, 1, r, lam) == STATE                  # no K
    G.build_rows(0, n // 2)
    assert adjoint_status(c, 0, 1, r, lam) == STATE                  # rows of part of the grid
    G.build_rows()
    assert adjoint_status(c, 0, 1, r, lam) == 0
    for e, k, rr, ll in ((2, 1, r, lam), (-1, 1, r, lam), (0, 0, r, lam), (0, 1, None, lam), (0, 1, r, None)):
        assert adjoint_status(c, e, k, rr, ll) == ARG, (e, k)
    M = binding.GpuMultiplet(synth.make_multiplet_scenario(0, 8, 6, 4, 4), "f64")
    M.build_rows()
    assert adjoint_status(M.ctx, 1, 1, rhs(M.n_el, 1), np.zeros((1, M.n_el))) == ARG
    # a zero right-hand side: lambda = 0, no steps, OK (also beside a nonzero one)
    z = np.zeros((2, n))
    z[1] = r[0]
    lam, steps, res = G.solve_adjoint(0, z)
    assert not lam[0].any() and steps[0] == 0 and res[0] == 0 and steps[1] > 0
    lam, steps, _ = G.solve_adjoint(0, np.zeros(n))
    assert not lam.any() and steps[0] == 0
    monkeypatch.setenv("B200RT_KRYLOV_MAXIT", "2")
    assert adjoint_status(c, 0, 1, r, lam) == NOT_DOMINANT
    assert "residual" in c.lib.b200rt_last_error(c.h).decode()


def facade_case(hb, synth, F):
    locs, dirs = synth.random_los(1500)
    F.add_observation(locs, dirs)
    F.generate_source_function(5e5, 200.0)
    w = np.random.default_rng(9).uniform(0.0, 1.0, len(locs))
    return locs, dirs, w


def test_facade(synth, binding):
    hb = importlib.import_module("3d_planetary_rt_model_b200.host_binding")
    F = hb.Pyobservation_fit(device=0)
    locs, dirs, w = facade_case(hb, synth, F)
    G = binding.GpuModel(synth.make_scenario(), "f64")              # the facade's model (test_facade_models.py)
    G.build_rows()
    G.solve()
    for e in range(2):
        lam = F.brightness_source_sensitivity(e, w)
        assert lam.shape == (F.n_vox,)
        assert rel_err(lam, G.brightness_source_sensitivity(locs, dirs, w, e), floor=1e-300) < 1e-5
    with pytest.raises(RuntimeError):
        F.brightness_source_sensitivity(0, w, hb.MODEL_H_PP)
    with pytest.raises(RuntimeError):
        F.brightness_source_sensitivity(0, w[:-1])


def test_fast_binding(synth, tmp_path):
    """the buffer-protocol .pyx path returns the facade's answer"""
    out = os.path.join(ROOT, "oracle", "_ref", "py_corona_sim_fast")
    if not (os.path.isdir(out) and any(f.startswith("py_corona_sim_gpu") and f.endswith(".so") for f in os.listdir(out))):
        pytest.skip("oracle/_ref/py_corona_sim_fast not built (needs B200RT_REFERENCE; python oracle/build_pyx.py)")
    dump = str(tmp_path / "lam.npy")
    code = f"""
import importlib, sys
import numpy as np
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {out!r})
import py_corona_sim_gpu as m
synth = importlib.import_module("3d_planetary_rt_model_b200.synth")
F = m.Pyobservation_fit_b200()
locs, dirs = synth.random_los(1500)
F.add_observation(locs, dirs)
F.generate_source_function(5e5, 200.0)
w = np.random.default_rng(9).uniform(0.0, 1.0, len(locs))
np.save({dump!r}, np.stack([F.brightness_source_sensitivity(e, w) for e in range(2)]))
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    hb = importlib.import_module("3d_planetary_rt_model_b200.host_binding")
    F = hb.Pyobservation_fit(device=0)
    _, _, w = facade_case(hb, synth, F)
    z = np.load(dump)
    for e in range(2):
        assert same_bits(z[e], F.brightness_source_sensitivity(e, w))
