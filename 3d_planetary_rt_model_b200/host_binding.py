"""ctypes binding of the C handles over the C++ observation_fit facade (host/capi.cpp, libb200rt_host.so).

The class below has the method names and argument lists of the reference's Cython class Pyobservation_fit
(python/py_corona_sim.pyx:176-562), plus brightness_batch and accessors for the solutions.  (The reference's own
.pyx also compiles unchanged against the facade: oracle/build_pyx.py.)"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libb200rt_host.so")
_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_vp = C.c_void_p

SIGNATURES = {
    "obsfit_last_error": (C.c_char_p, []),
    "obsfit_create": (_vp, [C.c_char_p, C.c_int]),
    "obsfit_create_ex": (_vp, [C.c_char_p, C.c_int, C.c_int]),
    "obsfit_destroy": (None, [_vp]),
    "obsfit_add_observation": (C.c_int, [_vp, C.c_int, _dp, _dp]),
    "obsfit_set_g_factor": (C.c_int, [_vp, C.c_double, C.c_double]),
    "obsfit_add_observation_ra_dec": (C.c_int, [_vp, _dp, C.c_int, _dp, _dp]),
    "obsfit_generate_source_function": (C.c_int, [_vp, C.c_double, C.c_double, C.c_char_p]),
    "obsfit_set_use_CO2_absorption": (C.c_int, [_vp, C.c_int]),
    "obsfit_set_CO2_exobase_density": (C.c_int, [_vp, C.c_double]),
    "obsfit_save_influence_matrix": (C.c_int, [_vp, C.c_char_p]),
    "obsfit_get": (C.c_int, [_vp, C.c_int, _dp]),
    "obsfit_source_function": (C.c_int, [_vp, C.c_int, _dp]),
    "obsfit_radial_boundaries": (C.c_int, [_vp, _dp]),
    "obsfit_brightness_batch": (C.c_int, [_vp, C.c_int, _dp, _dp, C.c_int, C.c_int, _dp, C.POINTER(C.c_double)]),
    "obsfit_atmosphere_tables": (C.c_int, [C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int, _dp, _dp]),
    "obsfit_generate_source_function_ex": (C.c_int, [_vp, C.c_double, C.c_double, C.c_char_p, C.c_char_p, C.c_int, C.c_int]),
    "obsfit_generate_source_function_lc": (C.c_int, [_vp, C.c_double, C.c_double, C.c_int, C.c_int]),
    "obsfit_generate_source_function_effv": (C.c_int, [_vp, C.c_double, C.c_double, C.c_int, C.c_int]),
    "obsfit_generate_source_function_variable_thermosphere": (C.c_int, [_vp] + [C.c_double] * 10 + [C.c_int, C.c_int]),
    "obsfit_generate_source_function_nH_asym": (C.c_int, [_vp, C.c_double, C.c_double, C.c_double, C.c_int]),
    "obsfit_generate_source_function_temp_asym": (C.c_int, [_vp, C.c_double, C.c_double, C.c_double, C.c_int]),
    "obsfit_generate_source_function_tabular_atmosphere": (C.c_int, [_vp, C.c_double, C.c_double, C.c_double, C.c_int, _dp, _dp,
                                                                     C.c_int, _dp, _dp, C.c_int, _dp, _dp, C.c_int, C.c_int, C.c_int]),
    "obsfit_O_1026_generate_source_function": (C.c_int, [_vp, C.c_double, C.c_double, C.c_double, C.c_char_p]),
    "obsfit_lyman_multiplet_generate_source_function": (C.c_int, [_vp, C.c_double, C.c_double, C.c_char_p]),
    "obsfit_lyman_singlet_generate_source_function": (C.c_int, [_vp, C.c_double, C.c_double, C.c_char_p]),
    "obsfit_save_influence_matrix_O_1026": (C.c_int, [_vp, C.c_char_p]),
    "obsfit_set_use_temp_dependent_sH": (C.c_int, [_vp, C.c_int, C.c_double]),
    "obsfit_set_sza_method": (C.c_int, [_vp, C.c_int]),
    "obsfit_set_tweak": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS"), C.c_double]),
    "obsfit_Tconv": (C.c_int, [_vp, C.c_int, C.c_double, C.POINTER(C.c_double)]),
    "obsfit_source_function_ex": (C.c_int, [_vp, C.c_int, C.c_int, _dp]),
    "obsfit_radial_boundaries_ex": (C.c_int, [_vp, C.c_int, _dp]),
    "obsfit_write_S_file": (C.c_int, [C.c_char_p, C.c_int, C.c_int, _dp, _dp, _dp, _dp, C.c_int, C.POINTER(C.c_char_p), _dp]),
    "obsfit_write_influence_file": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(C.c_char_p), _dp, C.c_int]),
    "obsfit_multiplet_source_function": (C.c_int, [_vp, C.c_int, _dp, C.c_int, C.POINTER(C.c_int)]),
    "obsfit_brightness_weights": (C.c_int, [_vp, C.c_int, C.c_int, C.POINTER(C.c_longlong), C.POINTER(C.c_int),
                                            C.POINTER(C.c_int)]),
    "obsfit_brightness_weights_get": (C.c_int, [_vp, _vp, _vp, _vp]),
}
MODEL_H, MODEL_D, MODEL_H_PP, MODEL_D_PP = 0, 1, 2, 3
_lib = None


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not built: run __graft_entry__.build()")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def write_S_file(fname, rb, pts_r, sb, pts_s, names, q):
    """the facade's save_S writer on plain arrays: q[n_em][8][n_vox] (order of the printed blocks)"""
    lib = load()
    q = np.ascontiguousarray(q, dtype=np.float64)
    nm = (C.c_char_p * len(names))(*[n.encode() for n in names])
    rc = lib.obsfit_write_S_file(os.fsencode(fname), len(rb), len(sb), np.ascontiguousarray(rb, dtype=np.float64),
                                 np.ascontiguousarray(pts_r, dtype=np.float64), np.ascontiguousarray(sb, dtype=np.float64),
                                 np.ascontiguousarray(pts_s, dtype=np.float64), len(names), nm, q)
    if rc != 0:
        raise RuntimeError(lib.obsfit_last_error().decode())


def write_influence_file(fname, names, K):
    """the facade's save_influence_matrix writer on plain arrays: K[n_em][n][n]"""
    lib = load()
    K = np.ascontiguousarray(K, dtype=np.float64)
    nm = (C.c_char_p * len(names))(*[n.encode() for n in names])
    if lib.obsfit_write_influence_file(os.fsencode(fname), len(names), nm, K, K.shape[-1]) != 0:
        raise RuntimeError(lib.obsfit_last_error().decode())


def atmosphere_tables(nH, nCO2, T, n_rb=40, n_sb=20, rmethod=0):
    """host only: the C++ chamb_diff_1d restatement -> (radial_boundaries[n_rb], tables[6][n_vox])"""
    lib = load()
    rb = np.zeros(n_rb)
    tabs = np.zeros((6, (n_rb - 1) * (n_sb - 1)))
    if lib.obsfit_atmosphere_tables(nH, nCO2, T, n_rb, n_sb, rmethod, rb, tabs) != 0:
        raise RuntimeError(lib.obsfit_last_error().decode())
    return rb, tabs


class Pyobservation_fit:
    n_emissions, n_rb, n_sb = 2, 40, 20
    n_vox = (n_rb - 1) * (n_sb - 1)

    def __init__(self, iph_table_fname="", device=-1, single_precision=False):
        self.lib = load()
        self.h = self.lib.obsfit_create_ex(os.fsencode(iph_table_fname), device, int(single_precision))
        if not self.h:
            raise RuntimeError(self.lib.obsfit_last_error().decode())
        self.n_obs = 0

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.obsfit_destroy(self.h)
            self.h = None

    def _ck(self, rc):
        if rc != 0:
            raise RuntimeError(self.lib.obsfit_last_error().decode())

    def add_observation(self, loc_arr, dir_arr):
        loc = np.ascontiguousarray(loc_arr, dtype=np.float64)
        d = np.ascontiguousarray(dir_arr, dtype=np.float64)
        self.n_obs = len(loc)
        self._ck(self.lib.obsfit_add_observation(self.h, self.n_obs, loc, d))

    def set_g_factor(self, g):
        self._ck(self.lib.obsfit_set_g_factor(self.h, float(g[0]), float(g[1])))

    def add_observation_ra_dec(self, mars_ecliptic_coords, ra, dec):
        self._ck(self.lib.obsfit_add_observation_ra_dec(self.h, np.ascontiguousarray(mars_ecliptic_coords, dtype=np.float64),
                                                        len(ra), np.ascontiguousarray(ra, dtype=np.float64),
                                                        np.ascontiguousarray(dec, dtype=np.float64)))

    def generate_source_function(self, nH, T, atmosphere_fname="", sourcefn_fname="", plane_parallel=False, deuterium=False):
        self._ck(self.lib.obsfit_generate_source_function_ex(self.h, nH, T, os.fsencode(atmosphere_fname), os.fsencode(sourcefn_fname),
                                                             int(plane_parallel), int(deuterium)))

    def generate_source_function_lc(self, nH, lc, plane_parallel=False, deuterium=False):
        self._ck(self.lib.obsfit_generate_source_function_lc(self.h, nH, lc, int(plane_parallel), int(deuterium)))

    def generate_source_function_effv(self, nH, effv, plane_parallel=False, deuterium=False):
        self._ck(self.lib.obsfit_generate_source_function_effv(self.h, nH, effv, int(plane_parallel), int(deuterium)))

    def generate_source_function_variable_thermosphere(self, nHexo, Texo, nCO2rmin, rexo, rmin, rmax, rmindiffusion, T_tropo,
                                                       r_tropo, shape_parameter, plane_parallel=False, deuterium=False):
        self._ck(self.lib.obsfit_generate_source_function_variable_thermosphere(
            self.h, nHexo, Texo, nCO2rmin, rexo, rmin, rmax, rmindiffusion, T_tropo, r_tropo, shape_parameter,
            int(plane_parallel), int(deuterium)))

    def generate_source_function_nH_asym(self, nH, Texo, asym, deuterium=False):
        self._ck(self.lib.obsfit_generate_source_function_nH_asym(self.h, nH, Texo, asym, int(deuterium)))

    def generate_source_function_temp_asym(self, nHavg, Tnoon, Tmidnight, deuterium=False):
        self._ck(self.lib.obsfit_generate_source_function_temp_asym(self.h, nHavg, Tnoon, Tmidnight, int(deuterium)))

    def generate_source_function_tabular_atmosphere(self, atm_dict, compute_exosphere=False, plane_parallel=False, deuterium=False):
        a = {k: np.ascontiguousarray(atm_dict[k], dtype=np.float64) for k in ("alt_nH", "log_nH", "alt_nCO2", "log_nCO2", "alt_Temp", "Temp")}
        self._ck(self.lib.obsfit_generate_source_function_tabular_atmosphere(
            self.h, atm_dict["rmin"], atm_dict["rexo"], atm_dict["rmax"], len(a["alt_nH"]), a["alt_nH"], a["log_nH"],
            len(a["alt_nCO2"]), a["alt_nCO2"], a["log_nCO2"], len(a["alt_Temp"]), a["alt_Temp"], a["Temp"],
            int(compute_exosphere), int(plane_parallel), int(deuterium)))

    def O_1026_generate_source_function(self, nO, T, solar_brightness_lyman_beta, sourcefn_fname=""):
        self._ck(self.lib.obsfit_O_1026_generate_source_function(self.h, nO, T, solar_brightness_lyman_beta, os.fsencode(sourcefn_fname)))

    def lyman_multiplet_generate_source_function(self, nH, T, sourcefn_fname=""):
        self._ck(self.lib.obsfit_lyman_multiplet_generate_source_function(self.h, nH, T, os.fsencode(sourcefn_fname)))

    def lyman_singlet_generate_source_function(self, nH, T, sourcefn_fname=""):
        self._ck(self.lib.obsfit_lyman_singlet_generate_source_function(self.h, nH, T, os.fsencode(sourcefn_fname)))

    def save_influence_matrix_O_1026(self, fname):
        self._ck(self.lib.obsfit_save_influence_matrix_O_1026(self.h, os.fsencode(fname)))

    def set_use_temp_dependent_sH(self, use=True, constant_temp_sH=-1.0):
        self._ck(self.lib.obsfit_set_use_temp_dependent_sH(self.h, int(use), constant_temp_sH))

    def set_sza_method_uniform(self):
        self._ck(self.lib.obsfit_set_sza_method(self.h, 0))

    def set_sza_method_uniform_cos(self):
        self._ck(self.lib.obsfit_set_sza_method(self.h, 1))

    def set_H_density_tweak(self, on, voxels=(), factor=1.0):
        self._ck(self.lib.obsfit_set_tweak(self.h, 0, int(on), len(voxels), np.ascontiguousarray(voxels, dtype=np.int32), factor))

    def set_H_temp_tweak(self, on, voxels=(), factor=1.0):
        self._ck(self.lib.obsfit_set_tweak(self.h, 1, int(on), len(voxels), np.ascontiguousarray(voxels, dtype=np.int32), factor))

    def _tconv(self, which, x):
        out = C.c_double(0)
        self._ck(self.lib.obsfit_Tconv(self.h, which, float(x), C.byref(out)))
        return out.value

    def lc_from_T(self, T):
        return self._tconv(0, T)

    def eff_from_T(self, T):
        return self._tconv(1, T)

    def T_from_lc(self, lc):
        return self._tconv(2, lc)

    def T_from_eff(self, eff):
        return self._tconv(3, eff)

    def set_use_CO2_absorption(self, use=True):
        self._ck(self.lib.obsfit_set_use_CO2_absorption(self.h, int(use)))

    def set_CO2_exobase_density(self, n):
        self._ck(self.lib.obsfit_set_CO2_exobase_density(self.h, n))

    def save_influence_matrix(self, fname):
        self._ck(self.lib.obsfit_save_influence_matrix(self.h, os.fsencode(fname)))

    def _get(self, which, rows=None):
        out = np.zeros((rows or self.n_emissions, self.n_obs))
        self._ck(self.lib.obsfit_get(self.h, which, out))
        return out

    def D_brightness(self):
        return self._get(6)

    def D_col_dens(self):
        return self._get(7)

    def tau_D_final(self):
        return self._get(8)

    def O_1026_brightness(self):
        return self._get(9, 6)

    def lyman_multiplet_brightness(self):
        return self._get(10)

    def lyman_singlet_brightness(self):
        return self._get(11)

    def multiplet_source_function(self, model):
        out = np.zeros(self.n_vox * 4)
        n = C.c_int(0)
        self._ck(self.lib.obsfit_multiplet_source_function(self.h, model, out, len(out), C.byref(n)))
        return out[:n.value].copy()

    def brightness(self):
        return self._get(0)

    def species_col_dens(self):
        return self._get(1)

    def tau_species_final(self):
        return self._get(2)

    def tau_absorber_final(self):
        return self._get(3)

    def iph_brightness_observed(self):
        return self._get(4)

    def iph_brightness_unextincted(self):
        return self._get(5)

    def source_function(self, e, which=MODEL_H):
        out = np.zeros(self.n_vox if which < 2 else self.n_rb - 1)
        self._ck(self.lib.obsfit_source_function_ex(self.h, e, which, out))
        return out

    def brightness_weights(self, e, which=MODEL_H):
        """line-of-sight weighting functions of emission e of model `which` for the current observations:
        (indptr, indices, data, shape); scipy.sparse.csr_matrix((data, indices, indptr), shape=shape) times
        source_function(e, which) is brightness()[e] without the IPH term"""
        nnz, nr, nc = C.c_longlong(0), C.c_int(0), C.c_int(0)
        self._ck(self.lib.obsfit_brightness_weights(self.h, e, which, C.byref(nnz), C.byref(nr), C.byref(nc)))
        indptr = np.zeros(nr.value + 1, np.int64)
        indices = np.zeros(max(nnz.value, 1), np.int32)
        data = np.zeros(max(nnz.value, 1))
        self._ck(self.lib.obsfit_brightness_weights_get(self.h, indptr.ctypes.data_as(_vp), indices.ctypes.data_as(_vp),
                                                        data.ctypes.data_as(_vp)))
        return indptr, indices[:nnz.value], data[:nnz.value], (nr.value, nc.value)

    def radial_boundaries(self, which=MODEL_H):
        out = np.zeros(self.n_rb)
        self._ck(self.lib.obsfit_radial_boundaries_ex(self.h, which, out))
        return out

    def brightness_batch(self, nH, T, contexts_per_gpu=4, n_gpus=-1):
        nH = np.ascontiguousarray(nH, dtype=np.float64)
        T = np.ascontiguousarray(T, dtype=np.float64)
        out = np.zeros((len(nH), self.n_emissions, self.n_obs))
        sec = C.c_double(0)
        self._ck(self.lib.obsfit_brightness_batch(self.h, len(nH), nH, T, contexts_per_gpu, n_gpus, out, C.byref(sec)))
        self.last_batch_seconds = sec.value
        return out
