"""Line-of-sight weights and the adjoint solve at the sizes where their kernels change code path.

test_los_weights.py and test_adjoint.py hold W and the adjoint to independent references on small grids.  The kernels
pick their path from the size of the problem, so this file repeats those checks where each switch flips: the multi-tile
row-pointer scan, several batches of lines of sight and the longest-first order of the value pass, W^T r without the
shared-memory copy of y, the structure bitmaps in global scratch, and the singlet GMRES (forward and adjoint) above the
size at which x leaves shared memory.  Each test asserts that its shape crosses the threshold it is about, computed from
the shape, so that a retuned constant fails here instead of silently leaving a path uncovered."""
import gc
import os

import numpy as np
import pytest

from test_los_weights import csr, mixed_los, random_S
from util import TOL, rel_err, same_bits

pytestmark = pytest.mark.gpu

SCAN_TILE = 4096                   # los_weights.cu: SCAN_THREADS * SCAN_ITEMS rows per tile of the row-pointer scan
LOS_ORDER_MIN = 4 * 148 * 4 * 32   # api_internal.hpp los_order_min(): 4 * NUM_SMS * 4 * 32 = 75,776
KRYLOV_MAX_N = 24576               # include/b200rt.h B200RT_KRYLOV_MAX_N
PROD = (100, 60, 24, 16)           # the bench grid: 5841 voxels
N_PROD = 100_000
FLOOR = {"f64": 1e-300, "f32": 1e-35}


def prod_scenario(synth, n_em):
    return synth.make_scenario(*PROD, n_em=n_em, rmethod=synth.RMETHOD_ALTITUDE, rmax=synth.rMars + 50000e5)


def same_csr(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and same_bits(a[2], b[2])


def stored_cols(W, r):
    indptr, indices, _ = W
    return indices[indptr[r]:indptr[r + 1]]


def check_structure(W, n_vox, n_em, ln):
    """the CSR checks of test_los_weights.test_structure; ln: boundary-list lengths of the lines of sight"""
    indptr, indices, data = W
    nnz = len(indices)
    assert indptr[0] == 0 and indptr[-1] == nnz
    d = np.diff(indptr)
    assert (d >= 0).all()
    assert ((indices >= 0) & (indices < n_vox)).all()
    inner = np.ones(nnz, bool)                    # every entry but the first of its row: strictly above its left one
    inner[indptr[:-1][d > 0]] = False
    assert (np.diff(indices, prepend=-1)[inner] > 0).all()
    assert (ln == 0).any()
    assert (d[ln == 0] == 0).all()                # grid misses: empty rows
    assert (d[ln > 1] > 0).all()
    assert data.shape == (n_em, nnz) and np.isfinite(data).all()


def check_entries(O, n_vox, locs, dirs, W, rows, prec):
    """Exact entries of `rows` against the oracle: for each voxel v stored in any of them, the oracle's brightness of
    those lines of sight with S = e_v is column v; then per row, S = 1 on every voxel the row does NOT store must give a
    brightness of exactly 0 (a dropped column cannot hide).  Row-scaled bar of test_entries_match_oracle."""
    cols = [stored_cols(W, r) for r in rows]
    union = np.unique(np.concatenate(cols))
    L, D = locs[rows], dirs[rows]
    Wo = np.zeros((len(rows), len(union)))
    ev = np.zeros(n_vox)
    for j, v in enumerate(union):
        ev[v] = 1.0
        O.set_sourcefn(0, ev)
        Wo[:, j] = O.brightness(L, D, 10)[1][0, 0]
        ev[v] = 0.0
    Wg = np.zeros_like(Wo)
    stored = np.zeros(Wo.shape, bool)
    indptr, _, data = W
    for k, r in enumerate(rows):
        pos = np.searchsorted(union, cols[k])
        Wg[k, pos] = data[0, indptr[r]:indptr[r + 1]]
        stored[k, pos] = True
    floor = FLOOR[prec]
    assert not (np.abs(Wo) > floor)[~stored].any(), "an oracle nonzero is not a stored entry"
    scale = np.maximum(np.abs(Wo).max(axis=1), floor)[:, None]
    assert (np.abs(Wg - Wo) / scale).max() < TOL[prec]
    for k, r in enumerate(rows):
        S = np.ones(n_vox)
        S[cols[k]] = 0.0
        O.set_sourcefn(0, S)
        assert O.brightness(locs[r:r + 1], dirs[r:r + 1], 10)[1][0, 0, 0] == 0.0, ("a column outside the row", r)


def check_products(G, W, e, n_los, seed=1):
    """W x and W^T r against scipy in FP64: the bar of test_los_weights.test_products"""
    rng = np.random.default_rng(seed)
    M = csr(W, e, G.n_vox)
    x, r = rng.uniform(-1, 1, G.n_vox), rng.uniform(-1, 1, n_los)
    y = G.ctx.los_weights_apply(e, x)
    assert np.abs(y - M @ x).max() <= 1e-13 * np.abs(M).dot(np.abs(x)).max()
    yt = G.ctx.los_weights_apply(e, r, transpose=True)
    assert np.abs(yt - M.T @ r).max() <= 1e-13 * np.abs(M.T).dot(np.abs(r)).max()


# ---------------------------------------------------------------- the multi-tile row-pointer scan
@pytest.fixture(scope="module")
def mid(synth, binding):
    scn = synth.make_scenario(20, 12, 6, 8, n_em=2, sza_T_contrast=0.1)
    G = binding.GpuModel(scn, "f64")
    yield scn, G
    G.ctx.close()


@pytest.mark.parametrize("n,tiles", [(4095, 1), (4096, 1), (4097, 2), (8192, 2), (8193, 3), (12289, 4)])
def test_multi_tile_scan(synth, mid, n, tiles):
    """W of N lines of sight in one build against the same lines of sight built in chunks of at most 3000 (each a
    one-tile scan) and stitched.  A row depends only on its own line of sight, accumulated in march order: identical"""
    scn, G = mid
    assert -(-n // SCAN_TILE) == tiles                # launch_lw_scan: tiles of the scan
    locs, dirs = mixed_los(synth, scn, n, seed=n)
    full = G.los_weights(locs, dirs, 10)
    assert full[0][n] == len(full[1]) == G.ctx.lw_nnz
    chunk = 3000
    assert chunk <= SCAN_TILE                         # every chunk is a one-tile scan
    ptr, ind, dat, off = [np.zeros(1, np.int64)], [], [], 0
    for a in range(0, n, chunk):
        p, i, d = G.los_weights(locs[a:a + chunk], dirs[a:a + chunk], 10)
        ptr.append(p[1:] + off)
        ind.append(i)
        dat.append(d)
        off += len(i)
    stitched = (np.concatenate(ptr), np.concatenate(ind), np.concatenate(dat, axis=1))
    assert np.array_equal(full[0], stitched[0]), "row pointers"
    assert np.array_equal(full[1], stitched[1]), "columns"
    assert same_bits(full[2], stitched[2]), "values"
    assert (np.diff(full[0]) == 0).any()              # empty rows (grid misses) are in the set


# ---------------------------------------------------------------- the bench grid, 10^5 lines of sight
@pytest.fixture(scope="module")
def prod_los(synth):
    scn = prod_scenario(synth, 1)
    return mixed_los(synth, scn, N_PROD, seed=13)


def per_ray_bytes(G, prec):
    """api_internal.hpp batch_capacity: boundary-list bytes per line of sight"""
    return G.ctx.cap * ((8 if prec == "f64" else 4) + 4) + 2 * 4


@pytest.mark.parametrize("n_em", [1, 2])
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_batches_and_order_are_invisible(synth, binding, monkeypatch, prod_los, prec, n_em):
    """one batch ordered (the default at 10^5 lines of sight), one batch unordered, five batches ordered and unordered:
    the same matrix to the bit"""
    locs, dirs = prod_los
    assert N_PROD >= LOS_ORDER_MIN                    # the default orders the value pass
    G = binding.GpuModel(prod_scenario(synth, n_em), prec)
    per_batch = N_PROD // 5
    batches = -(-N_PROD // per_batch)
    settings = {"default": (None, None, 1, True), "unordered": (None, "1000000000", 1, False),
                "batched ordered": (str(per_ray_bytes(G, prec) * per_batch), "1000", batches, True),
                "batched unordered": (str(per_ray_bytes(G, prec) * per_batch), "1000000000", batches, False)}
    assert batches >= 4
    ref = None
    for name, (scratch, order_min, n_batches, ordered) in settings.items():
        for var, val in (("B200RT_SCRATCH_BYTES", scratch), ("B200RT_LOS_ORDER_MIN", order_min)):
            if val is None:
                monkeypatch.delenv(var, raising=False)
            else:
                monkeypatch.setenv(var, val)
        W = G.los_weights(locs, dirs, 10)
        # batches: the structure pass traverses each batch, and a batched build traverses each again for the values
        assert G.ctx.kernel_ms(binding.PH_TRAVERSE)[1] == (1 if n_batches == 1 else 2 * n_batches), name
        assert G.ctx.kernel_ms(binding.PH_ORDER)[1] == (3 * n_batches if ordered else 0), name
        assert W[2].shape[0] == n_em
        if ref is None:
            ref = W
            continue
        assert same_csr(ref, W), name
    G.ctx.close()


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_production_size_against_oracle(synth, binding, oraclebind, prod_los, prec):
    locs, dirs = prod_los
    scn = prod_scenario(synth, 1)
    G = binding.GpuModel(scn, prec)
    W = G.los_weights(locs, dirs, 10)
    n = len(locs)
    check_products(G, W, 0, n)
    S = random_S(G.n_vox, 0, seed=41)
    WS = csr(W, 0, G.n_vox) @ S
    G.set_sourcefn(0, S)
    _, b = G.brightness(locs, dirs, 10)
    ref = b[0, 0]
    assert np.abs(WS - ref).max() / np.abs(ref).max() < (1e-12 if prec == "f64" else 1e-4)
    G.ctx.close()

    O = oraclebind.OracleModel(scn, prec)
    O.set_sourcefn(0, S)
    rng = np.random.default_rng(43)
    sample = np.sort(rng.choice(n, 300, replace=False))
    bo = O.brightness(locs[sample], dirs[sample], 10)[1][0, 0]
    assert np.abs(WS[sample] - bo).max() / np.abs(bo).max() < TOL[prec]

    # 8 rows: the longest, one that re-enters a voxel it left, and 6 seeded non-empty ones
    lengths = np.diff(W[0])
    ln, _, ent, _, _ = O.traverse_los(locs, dirs)
    start = np.concatenate([[0], np.cumsum(ln)])
    reenter = next(i for i in range(n) if len(np.unique(ent[start[i]:start[i + 1]])) < ln[i] and lengths[i] > 0)
    rows = [int(np.argmax(lengths)), reenter]
    rows += [int(r) for r in rng.choice(np.flatnonzero(lengths > 0), 6, replace=False) if r not in rows]
    check_entries(O, G.n_vox, locs, dirs, W, rows, prec)


# ---------------------------------------------------------------- a singlet grid of 16,510 voxels
@pytest.fixture(scope="module")
def singlet16k(synth, binding):
    scn = synth.make_scenario(128, 131, 12, 8, n_em=1, sza_T_contrast=0.1)
    G = binding.GpuModel(scn, "f64")
    assert scn.n_rb <= 128                            # traverse.cu: every traversal on the fast path
    assert 16384 < G.n_vox <= KRYLOV_MAX_N            # above the GMRES's former capacity, within the current one
    # kry_iterate stages x (n * 8 bytes) in each CTA only where a grid of ceil(n / KRY_SLICE) CTAs (KRY_SLICE = 96) fits
    # beside it: 172 CTAs need two per SM of the 148, and two copies of x exceed an SM's 228 kB.  So x comes through L2
    assert -(-G.n_vox // 96) > 148 and 2 * G.n_vox * 8 > 228 * 1024
    G.build_rows()
    K = G.K(0)
    yield scn, G, K
    G.ctx.close()


def test_16k_rows_match_oracle(singlet16k, oraclebind):
    scn, G, K = singlet16k
    O = oraclebind.OracleModel(scn, "f64")
    v0, stride = 17, 1651
    O.build_rows(v0, scn.n_vox, stride)
    Ko = O.K(0)
    for v in range(v0, scn.n_vox, stride):
        a = np.where(np.abs(Ko[v]) > 1e-290, Ko[v], 0.0)
        b = np.where(np.abs(K[v]) > 1e-290, K[v], 0.0)
        assert np.array_equal(a != 0, b != 0), v
        assert rel_err(a, b) < TOL["f64"], v


def test_16k_forward_solve(singlet16k, monkeypatch):
    scn, G, K = singlet16k
    w = float(scn.em_scalars[0][0])
    monkeypatch.delenv("B200RT_SOLVER", raising=False)
    G.solve()
    assert G.ctx.last_solve_steps() > 0               # b200rt_solve took the GMRES
    v = G.vectors(0)
    S, S0 = v["S"], v["S0"]
    assert np.abs(S - w * (K @ S) - S0).max() / np.abs(S0).max() <= 1e-12
    monkeypatch.setenv("B200RT_SOLVER", "lu")
    G.solve()
    assert np.abs(S - G.vectors(0)["S"]).max() <= 1e-10 * np.abs(S).max()


def test_16k_adjoint(singlet16k, monkeypatch):
    scn, G, K = singlet16k
    w = float(scn.em_scalars[0][0])
    monkeypatch.delenv("B200RT_SOLVER", raising=False)
    G.solve()
    assert G.ctx.last_solve_steps() > 0
    v = G.vectors(0)
    r = np.random.default_rng(31).uniform(-1.0, 1.0, (3, G.n_vox))
    lam, steps, _ = G.solve_adjoint(0, r)
    assert (steps > 0).all()
    # (K^T lam)_i = sum_j K[j, i] lam_j
    assert (np.abs(lam - w * (lam @ K) - r).max(axis=1) / np.abs(r).max(axis=1) <= 1e-12).all()
    for k in range(3):
        assert abs(r[k] @ v["S"] - lam[k] @ v["S0"]) <= 1e-10 * np.abs(r[k]).dot(np.abs(v["S"]))
    monkeypatch.setenv("B200RT_KRYLOV_FUSED", "0")    # the per-step launches, no preconditioner
    lam0, _, _ = G.solve_adjoint(0, r)
    assert np.abs(lam - lam0).max() <= 1e-10 * np.abs(lam).max()


def test_16k_weights(synth, singlet16k):
    scn, G, K = singlet16k
    assert G.n_vox * 8 > 96 * 1024                    # launch_lw_apply: W^T r without the shared-memory copy of y
    G.solve()
    locs, dirs = mixed_los(synth, scn, 500, seed=37)
    W = G.los_weights(locs, dirs, 10)
    check_products(G, W, 0, len(locs), seed=3)
    S = G.vectors(0)["S"]
    _, b = G.brightness(locs, dirs, 10)
    WS = csr(W, 0, G.n_vox) @ S
    assert np.abs(WS - b[0, 0]).max() <= 1e-12 * np.abs(b[0, 0]).max()
    wl = np.random.default_rng(3).uniform(0.0, 1.0, len(locs))
    lam = G.brightness_source_sensitivity(locs, dirs, wl, 0)
    lhs = wl @ b[0, 0]
    assert lhs > 0
    assert abs(lhs - lam @ G.vectors(0)["S0"]) <= 1e-11 * lhs


# ---------------------------------------------------------------- structure bitmaps in global scratch: 65,659 voxels
def resident_bytes():
    with open("/proc/self/statm") as f:
        return int(f.read().split()[1]) * os.sysconf("SC_PAGE_SIZE")


def free_device_bytes():
    import torch
    return torch.cuda.mem_get_info(0)[0]


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_global_bitmaps(synth, binding, oraclebind, prec):
    scn = synth.make_scenario(128, 518, 4, 4, n_em=1, sza_T_contrast=0.1)
    n_vox = scn.n_vox
    assert -(-n_vox // 32) * 4 * 8 > 64 * 1024        # los_weights.cu LW_SMEM_BITMAP_MAX: bitmaps in global scratch
    # b200rt_set_singlet reserves the FP64 K of the grid (n_vox^2 doubles, 34.5 GB) although no influence build runs
    free = free_device_bytes()
    if free < 40e9:
        pytest.skip(f"needs 40 GB of free device memory for the {n_vox}-voxel grid's K; {free / 1e9:.1f} GB free")
    G = binding.GpuModel(scn, prec)
    try:
        locs, dirs = mixed_los(synth, scn, 2000, seed=19)
        W = G.los_weights(locs, dirs, 10)
        check_structure(W, n_vox, 1, G.ctx.traverse_los()[0])
        S = random_S(n_vox, 0, seed=47)
        WS = csr(W, 0, n_vox) @ S
        G.set_sourcefn(0, S)
        _, b = G.brightness(locs, dirs, 10)
        assert np.abs(WS - b[0, 0]).max() / np.abs(b[0, 0]).max() < (1e-12 if prec == "f64" else 1e-4)
    finally:
        G.ctx.close()
        del G
        gc.collect()
    rss = resident_bytes()
    O = oraclebind.OracleModel(scn, prec)
    O.set_sourcefn(0, S)
    bo = O.brightness(locs, dirs, 10)[1][0, 0]
    assert np.abs(WS - bo).max() / np.abs(bo).max() < TOL[prec]
    lengths = np.diff(W[0])
    rng = np.random.default_rng(53)
    rows = [int(np.argmax(lengths))]
    rows += [int(r) for r in rng.choice(np.flatnonzero(lengths > 0), 5, replace=False) if r not in rows]
    check_entries(O, n_vox, locs, dirs, W, rows, prec)
    assert resident_bytes() - rss < 1e9       # the oracle's K (n_vox^2 reals, calloc'd) is reserved, never touched
