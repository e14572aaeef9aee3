"""Stored results of the comparisons with the reference's own source (test_oracle_vs_ref, test_plane_parallel,
test_multiplet, test_file_formats), so that the oracle is held to them where the reference build (oracle/_ref) is absent.

Each *_case function runs one of those comparisons on one model (refbind / multbind reference or oracle: same method
names) and returns what was compared: arrays compared bit for bit are kept as SHA-256 digests of their bytes, source
functions (compared to a tolerance: two different LUs) in full.  tests/golden/make_ref_pins.py writes them to
tests/golden/ref_pins.json and ref_pins_S.npz; the *_pins tests recompute them with the oracle and compare."""
import hashlib
import json
import os
import tempfile

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DIGESTS, SOURCEFNS = os.path.join(GOLDEN, "ref_pins.json"), os.path.join(GOLDEN, "ref_pins_S.npz")

SINGLET_SHAPES = [(8, 6, 4, 4), (12, 8, 5, 6), (20, 12, 6, 8)]
PP_SHAPES = [(8, 4), (12, 5), (40, 7), (40, 6)]
MULT_SHAPES = [(8, 6, 4, 4), (12, 8, 5, 6)]
MULT_KINDS = [0, 1, 2]
FILE_CASES = [((8, 6, 4, 4), 2), ((12, 8, 5, 6), 1)]


def digest(a):
    """the first 64 bits of the SHA-256 of the array's bytes as float64 (integers as int64), with its shape"""
    a = np.asarray(a)
    a = np.ascontiguousarray(a, dtype=np.int64 if a.dtype.kind in "iub" else np.float64)
    return hashlib.sha256(repr(a.shape).encode() + a.tobytes()).hexdigest()[:16]


def _lists(out, pre, lists):
    for k, v in zip(("len", "eb", "ent", "dist"), lists):
        out[f"{pre}_{k}"] = v


def singlet_case(synth, M, S=None):
    """test_oracle_vs_ref.test_oracle_matches_reference on one model.  S: the source functions to set before the
    brightness (the reference's, as the live test does); None = the model's own.  -> (compared arrays, own S, residuals)"""
    out = {"grid_" + k: v for k, v in M.grid().items() if k != "radial_boundaries"}
    for e in range(2):
        out.update({f"arr{e}_{k}": v for k, v in M.arrays(e).items()})
    _lists(out, "vr", M.traverse_voxel_rays())
    out["n_steps"] = M.build_rows()[1]
    for e in range(2):
        out[f"K{e}"] = M.K(e)
        v = M.vectors(e)
        out.update({f"vec{e}_{k}": v[k] for k in ("S0", "tau_species_ss", "tau_absorber_ss")})
    res = M.solve()
    own = [M.vectors(e)["S"] for e in range(2)]
    for e in range(2):
        M.set_sourcefn(e, own[e] if S is None else S[e])
    for j, (locs, dirs) in enumerate((synth.fake_image(30 * synth.rMars, 30, 24), synth.random_los(600))):
        t = M.traverse_los(locs, dirs)
        _lists(out, f"los{j}", t[:4])
        out[f"los{j}_rayscal"] = t[4]
        for nsub in (10, 0, 3):
            out[f"los{j}_b{nsub}"] = M.brightness(locs, dirs, nsub)[1]
    return out, own, res


def grid_D_case(synth, M):
    """test_oracle_vs_ref.test_default_grid_D: the 40x20x7x12 grid, 2 emissions"""
    out = {}
    _lists(out, "vr", M.traverse_voxel_rays(0, 200))
    M.build_rows()
    M.solve()
    out.update({f"vec{e}_S0": M.vectors(e)["S0"] for e in range(2)})
    return out, [M.vectors(e)["S"] for e in range(2)]


def pp_case(M):
    """test_plane_parallel.test_oracle_matches_reference_pp on one model"""
    g = M.grid()
    out = {"grid_" + k: g[k] for k in ("pts_radii", "ray_theta", "ray_domega")}
    for e in range(2):
        out.update({f"arr{e}_{k}": v for k, v in M.arrays(e).items()})
    _lists(out, "vr", M.traverse_voxel_rays())
    out["n_steps"] = M.build_rows()[1]
    for e in range(2):
        out[f"K{e}"] = M.K(e)
        v = M.vectors(e)
        out.update({f"vec{e}_{k}": v[k] for k in ("S0", "tau_species_ss", "tau_absorber_ss")})
    res = M.solve()
    return out, [M.vectors(e)["S"] for e in range(2)], res


def mult_case(synth, M, S=None):
    """test_multiplet.test_oracle_matches_reference on one model (RefMultiplet / OracleMultiplet)"""
    out = {"dims": [M.n_lines, M.n_mult, M.n_lower, M.n_upper, M.n_lambda]}
    out.update({"const_" + k: v for k, v in M.constants().items()})
    out["lineshape"] = [M.lineshape(line, i, T) for line in range(M.n_lines) for i in range(M.n_lambda)
                        for T in (131.7, 200.0, 263.1)]
    out.update({"arr_" + k: v for k, v in M.arrays().items()})
    out["n_steps"] = M.build_rows()[1]
    out["K"] = M.K()
    v = M.vectors()
    out.update({"vec_" + k: v[k] for k in ("S0", "tau_species_ss", "tau_absorber_ss")})
    res = M.solve()
    own = M.vectors()["S"]
    M.set_sourcefn(own if S is None else S)
    for j, (locs, dirs) in enumerate((synth.fake_image(30 * synth.rMars, 30, 10), synth.random_los(300))):
        for nsub in (10, 0, 3):
            out.update({f"los{j}_b{nsub}_{k}": v for k, v in M.brightness(locs, dirs, nsub).items()})
    return out, own, res


def mult_grid_D_case(synth, M):
    """test_multiplet.test_oracle_matches_reference_default_grid: O I 102.6 on 40x20x7x12, every 97th source voxel"""
    scn_n_vox = M.n_vox
    _, ns = M.build_rows(0, scn_n_vox, 97)
    rows = np.concatenate([np.arange(v * M.n_upper, (v + 1) * M.n_upper) for v in range(0, scn_n_vox, 97)])
    return {"n_steps": ns, "K_rows": M.K()[rows], "S0_rows": M.vectors()["S0"][rows]}


def file_case(scn, M, hb):
    """test_file_formats.test_save_S_and_influence_bytes: the facade's writers on a solved model's arrays (the reference's
    save_S / save_influence wrote the same bytes from the same arrays) -> the bytes of both files"""
    M.build_rows()
    M.solve()
    g = M.grid()
    names = [f"emission {e}" for e in range(scn.n_em)]
    q = np.zeros((scn.n_em, 8, scn.n_vox))
    K = np.zeros((scn.n_em, scn.n_vox, scn.n_vox))
    for e in range(scn.n_em):
        a, v = M.arrays(e), M.vectors(e)
        q[e] = [a["density"], v["tau_species_ss"], float(scn.em_scalars[e][2]) * np.sqrt(a["T_ratio"]), scn.vox_in[4],
                v["tau_absorber_ss"], np.full(scn.n_vox, float(scn.abs_sigma[e])), v["S0"], v["S"]]
        K[e] = M.K(e)
    with tempfile.TemporaryDirectory() as d:
        pS, pK = os.path.join(d, "S.dat"), os.path.join(d, "K.dat")
        hb.write_S_file(pS, scn.rb, g["pts_radii"], g["sza_boundaries"], g["pts_sza"], names, q)
        hb.write_influence_file(pK, names, K)
        return {"S_file": np.frombuffer(open(pS, "rb").read(), np.uint8),
                "K_file": np.frombuffer(open(pK, "rb").read(), np.uint8)}


class Pins:
    """digests[case][name] and sourcefns[case][e]; `source` says which model wrote them"""

    def __init__(self, source=None):
        self.source, self.digests, self.sourcefns = source, {}, {}

    @classmethod
    def load(cls):
        d = json.load(open(DIGESTS))
        p = cls(d["source"])
        p.digests = d["digests"]
        z = np.load(SOURCEFNS)
        for k in sorted(z.files):                                   # "<case>/<e>", fewer than ten emissions
            p.sourcefns.setdefault(k.rsplit("/", 1)[0], []).append(z[k])
        return p

    def store(self, case, out, S=()):
        self.digests[case] = {k: digest(v) for k, v in sorted(out.items())}
        if len(S):
            self.sourcefns[case] = [np.asarray(s, dtype=np.float64) for s in S]

    def save(self):
        with open(DIGESTS, "w") as f:
            json.dump({"source": self.source, "digests": self.digests}, f, indent=0, sort_keys=True)
            f.write("\n")
        np.savez_compressed(SOURCEFNS, **{f"{c}/{e}": s for c, S in self.sourcefns.items() for e, s in enumerate(S)})

    def check(self, case, out):
        """every array of `out` against the digest stored for `case`; the set of names must match too"""
        stored = self.digests[case]
        assert sorted(stored) == sorted(out), (case, set(stored) ^ set(out))
        bad = [k for k in out if digest(out[k]) != stored[k]]
        assert not bad, (case, bad)
