"""bench.py --dump-outputs: what it writes, from a stand-in for the context (CPU) and from a real run (gpu marker)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from util import TOL_AUX, UNDERFLOW, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOS_KEYS = ("brightness", "tau_species_final", "tau_absorber_final", "species_col_dens")


class FakeContext:
    def __init__(self, n_vox, n_los):
        self.n_vox, self.n_los = n_vox, n_los
        self.los = {k: np.arange(n_los, dtype=np.float64)[None, :] + q for q, k in enumerate(LOS_KEYS)}

    def solution(self, e):
        return {k: np.full(self.n_vox, float(q)) for q, k in enumerate(("S", "S0", "tau_species_ss", "tau_absorber_ss"))}

    def los_download(self):
        return self.los


def dump(tmp_path, n_vox, n_los):
    K = torch.arange(n_vox * n_vox, dtype=torch.float64).reshape(n_vox, n_vox)
    bench.dump_outputs(str(tmp_path), FakeContext(n_vox, n_los), K, n_vox)
    return K.numpy(), {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}


def test_small_outputs_are_written_whole(tmp_path):
    K, out = dump(tmp_path, 40, 1000)
    assert sorted(out) == sorted(("S", "S0", "tau_species_ss", "tau_absorber_ss", "influence_matrix_rows") + LOS_KEYS)
    assert all(a.dtype == np.float64 for a in out.values())
    assert np.array_equal(out["influence_matrix_rows"], K)
    assert np.array_equal(out["brightness"], np.arange(1000.0))


def test_large_outputs_are_a_fixed_sample_within_64_mb(tmp_path):
    n_vox, n_los = 1000, bench.DUMP_MAX_LOS + 12345
    assert (bench.DUMP_K_ROWS + 4) * 5841 * 8 + 4 * bench.DUMP_MAX_LOS * 8 <= 64 << 20        # the bench's 5841 voxels
    (tmp_path / "a").mkdir()
    K, out = dump(tmp_path / "a", n_vox, n_los)
    rows = out["influence_matrix_rows"]
    assert rows.shape == (bench.DUMP_K_ROWS, n_vox)
    assert np.array_equal(rows, K[(rows[:, 0] // n_vox).astype(int)])        # whole rows of K
    b = out["brightness"]
    assert b.shape == (bench.DUMP_MAX_LOS,) and np.all(np.diff(b) > 0)          # distinct lines of sight, in order
    for q, k in enumerate(LOS_KEYS):
        assert np.array_equal(out[k], b + q)                                     # the same lines of sight in every file
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    (tmp_path / "b").mkdir()
    _, again = dump(tmp_path / "b", n_vox, n_los)
    assert all(np.array_equal(out[k], again[k]) for k in out)                    # same sample from run to run


def test_bad_arguments_are_refused():
    for args, env in ((["--steps", "0"], {}), (["--dump-outputs", "x"], {"WORLD_SIZE": "2"})):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                           env=dict(os.environ, **env), timeout=120)
        assert r.returncode == 2 and "error:" in r.stderr


@pytest.mark.gpu
def test_bench_dumps_what_its_last_step_computed(tmp_path, synth, oraclebind):
    """the real run: K rows and S0 against the oracle's rows, S against (I - w K) S = S0 on those rows, the line-of-sight
    results against the oracle given the dumped S"""
    n_los = 5000
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--n-los", str(n_los),
                        "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    d = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    scn, locs, dirs = bench.make_workload(synth, n_los)
    rows = np.sort(np.random.default_rng(bench.DUMP_SEED).choice(scn.n_vox, bench.DUMP_K_ROWS, replace=False))
    O = oraclebind.OracleModel(scn, "f64")
    for v in rows:
        O.build_rows(int(v), int(v) + 1)
    Ko, Kg = O.K(0)[rows], d["influence_matrix_rows"]
    assert np.array_equal(np.abs(Ko) > 1e-290, np.abs(Kg) > 1e-290)
    assert rel_err(np.where(np.abs(Ko) > 1e-290, Ko, 0.0), np.where(np.abs(Kg) > 1e-290, Kg, 0.0)) < 1e-6
    assert rel_err(O.vectors(0)["S0"][rows], d["S0"][rows], floor=UNDERFLOW["f64"]) < 1e-6
    S, w = d["S"], float(scn.em_scalars[0][0])
    assert np.abs(S[rows] - w * Kg @ S - d["S0"][rows]).max() < 1e-10 * np.abs(S).max()
    O.set_sourcefn(0, S)
    _, b = O.brightness(locs[:500], dirs[:500], 10)
    for q, k in enumerate(LOS_KEYS):
        assert d[k].shape == (n_los,)
        assert np.array_equal(b[0, q] == -1, d[k][:500] == -1), k
        assert rel_err(b[0, q], d[k][:500], floor=1e-300) < TOL_AUX["f64"], k
