"""ctypes binding of the C ABI in include/b200rt.h (libb200rt.so).

This is the same thin stub a maintainer of the reference would add on the Python
side (INTEGRATION.md shows the C++ one).  There is no fallback of any kind: if the
shared library is missing, or no CUDA device is visible, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libb200rt.so")

F64, F32 = 0, 1
ROW_MAJOR, COL_MAJOR = 0, 1
PH_TRAVERSE, PH_INFLUENCE, PH_SOLVE, PH_BRIGHTNESS, PH_IPH, PH_ORDER = 0, 1, 2, 3, 4, 5

_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_fp = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_vp = C.c_void_p

# every symbol include/b200rt.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "b200rt_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(_vp)]),
    "b200rt_destroy": (C.c_int, [_vp]),
    "b200rt_last_error": (C.c_char_p, [_vp]),
    "b200rt_device_count": (C.c_int, []),
    "b200rt_create_multi": (C.c_int, [C.c_int, _vp, C.c_int, C.POINTER(_vp)]),
    "b200rt_group_size": (C.c_int, [_vp]),
    "b200rt_set_grid_sph": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int] + [_dp] * 7),
    "b200rt_make_grid_sph": (C.c_int, [C.c_int] * 5 + [_dp, C.c_int, C.c_int] + [_dp] * 6),
    "b200rt_set_grid_pp": (C.c_int, [_vp, C.c_int, C.c_int] + [_dp] * 4),
    "b200rt_make_grid_pp": (C.c_int, [C.c_int] * 3 + [_dp] * 4),
    "b200rt_fold_rays": (C.c_int, [C.c_int, C.c_int] + [_dp] * 3 + [_ip, C.POINTER(C.c_int)]),
    "b200rt_set_singlet": (C.c_int, [_vp, C.c_int, C.c_int] + [C.c_double] * 4 + [_dp] * 8),
    "b200rt_set_g_factor": (C.c_int, [_vp, C.c_int, C.c_double]),
    "b200rt_influence_ranges": (C.c_int, [_vp, C.c_int, np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS"),
                                          np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")]),
    "b200rt_ipc_export_influence": (C.c_int, [_vp, C.c_int, C.c_char_p]),
    "b200rt_ipc_open": (C.c_int, [_vp, C.c_char_p, C.POINTER(C.c_void_p)]),
    "b200rt_ipc_close": (C.c_int, [_vp, _vp]),
    "b200rt_set_row_sink": (C.c_int, [_vp, C.c_int, _vp]),
    "b200rt_solve_exchange": (C.c_int, [_vp, C.POINTER(C.c_void_p), C.c_char_p]),
    "b200rt_solve_distributed": (C.c_int, [_vp, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "b200rt_last_solve_steps": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "b200rt_multiplet_desc_init": (C.c_int, [C.c_int, C.c_int, _vp]),
    "b200rt_set_multiplet": (C.c_int, [_vp, _vp] + [_dp] * 6),
    "b200rt_generate_S": (C.c_int, [_vp]),
    "b200rt_influence": (C.c_int, [_vp, C.c_int, C.c_int]),
    "b200rt_solve": (C.c_int, [_vp]),
    "b200rt_last_step_count": (C.c_int, [_vp, C.POINTER(C.c_longlong)]),
    "b200rt_last_substep_count": (C.c_int, [_vp, C.POINTER(C.c_longlong)]),
    "b200rt_get_solution": (C.c_int, [_vp] + [C.c_int] + [_vp] * 4),
    "b200rt_get_influence": (C.c_int, [_vp, C.c_int, C.c_int, _dp]),
    "b200rt_set_sourcefn": (C.c_int, [_vp, C.c_int, _dp]),
    "b200rt_last_residual": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_double)]),
    "b200rt_influence_dev": (C.c_int, [_vp, C.c_int] + [C.POINTER(_vp)] * 4),
    "b200rt_sourcefn_dev": (C.c_int, [_vp, C.c_int, C.POINTER(_vp)]),
    "b200rt_los_from_MSO": (C.c_int, [C.c_int, C.c_int] + [_dp] * 11),
    "b200rt_brightness": (C.c_int, [_vp, C.c_int] + [_dp] * 9 + [C.c_int] + [_vp] * 4),
    "b200rt_los_upload": (C.c_int, [_vp, C.c_int] + [_dp] * 9),
    "b200rt_brightness_resident": (C.c_int, [_vp, C.c_int]),
    "b200rt_los_download": (C.c_int, [_vp] + [_vp] * 4),
    "b200rt_iph_load_table": (C.c_int, [_vp, C.c_char_p]),
    "b200rt_iph_set_table": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_float] + [_fp] * 7),
    "b200rt_iph_background": (C.c_int, [_vp] + [C.c_float] * 4 + [C.c_int, _fp, _fp, _fp, _fp, _vp]),
    "b200rt_iph_model": (C.c_int, [_vp, C.c_double, _dp, C.c_int, _dp, _dp, _dp]),
    "b200rt_iph_extinction": (C.c_int, [C.c_int, _dp, _dp, _dp]),
    "b200rt_traverse_voxel_rays": (C.c_int, [_vp, C.c_int, C.c_int, C.c_longlong, _ip, _ip, _ip, _dp,
                                             C.POINTER(C.c_longlong)]),
    "b200rt_traverse_los": (C.c_int, [_vp, C.c_longlong, _ip, _ip, _ip, _dp, C.POINTER(C.c_longlong)]),
    "b200rt_last_kernel_ms": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "b200rt_synchronize": (C.c_int, [_vp]),
    "b200rt_measure_fp64_peaks": (C.c_int, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}

MAX_LINES = 6


class MultipletDesc(C.Structure):
    """b200rt_multiplet_desc (include/b200rt.h)"""
    _fields_ = [("kind", C.c_int), ("n_lines", C.c_int), ("n_multiplets", C.c_int), ("n_lower", C.c_int),
                ("n_upper", C.c_int), ("n_lambda", C.c_int),
                ("multiplet_index", C.c_int * MAX_LINES), ("lower_level_index", C.c_int * MAX_LINES),
                ("upper_level_index", C.c_int * MAX_LINES),
                ("line_sigma_total", C.c_double * MAX_LINES), ("line_A", C.c_double * MAX_LINES),
                ("absorber_xsec", C.c_double * MAX_LINES), ("upper_state_decay_rate", C.c_double * MAX_LINES),
                ("offset", C.c_double * MAX_LINES), ("norm", C.c_double * MAX_LINES), ("weight", C.c_double * MAX_LINES),
                ("T_ref", C.c_double), ("lambda_max", C.c_double),
                ("solar_flux", C.c_double * MAX_LINES), ("pumped", C.c_int * MAX_LINES)]


_lib = None


def load():
    """dlopen libb200rt.so and type every entry point; raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("B200RT_LIB", LIB_PATH)     # development aid: an experimental build of the same library
    if not os.path.exists(path):
        raise RuntimeError(f"{path} not built: run __graft_entry__.build() (there is no CPU fallback)")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class B200RTError(RuntimeError):
    pass


def fold_rays(precision, ray_theta, ray_phi, ray_domega):
    """b200rt_fold_rays (host only): (rep, n_marched) -- rep[k] is the ray whose march stands for ray k in an influence
    build (k itself for a marched ray; the lower index of a mirror pair)"""
    lib = load()
    t, p, d = (np.ascontiguousarray(a, dtype=np.float64) for a in (ray_theta, ray_phi, ray_domega))
    rep = np.zeros(len(t), dtype=np.int32)
    n = C.c_int(0)
    rc = lib.b200rt_fold_rays(precision, len(t), t, p, d, rep, C.byref(n))
    if rc != 0:
        raise B200RTError(f"b200rt_fold_rays: status {rc}")
    return rep, n.value


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_vp)


class Context:
    """One b200rt_ctx: one GPU (device=...) or several GPUs of this process behind one handle (devices=[...] or
    devices="all": b200rt_create_multi).  Method names follow the reference's RT_grid where one exists."""

    def __init__(self, device: int = 0, precision: int = F64, devices=None):
        self.lib = load()
        self.h = _vp()
        if devices is None:
            rc = self.lib.b200rt_create(device, precision, C.byref(self.h))
        elif isinstance(devices, str):     # "all"
            rc = self.lib.b200rt_create_multi(0, None, precision, C.byref(self.h))
        else:
            ids = (C.c_int * len(devices))(*[int(d) for d in devices])
            rc = self.lib.b200rt_create_multi(len(devices), C.cast(ids, _vp), precision, C.byref(self.h))
        if rc != 0:
            raise B200RTError(f"b200rt_create(device={device}, devices={devices}) failed with status {rc}: no usable "
                              "CUDA device (this library has no CPU path)")
        self.n_devices = self.lib.b200rt_group_size(self.h)
        self.precision = precision
        self.n_vox = 0
        self.n_em = 0
        self.n_los = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.b200rt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise B200RTError(f"status {rc}: {self.lib.b200rt_last_error(self.h).decode()}")

    # ---- geometry
    def make_grid(self, n_rb, n_sb, n_theta, n_phi, rb, szamethod, raymethod):
        n_rays = n_theta * n_phi
        out = dict(radial_boundaries=np.ascontiguousarray(rb, dtype=np.float64),
                   sza_boundaries=np.zeros(n_sb), pts_radii=np.zeros(n_rb - 1), pts_sza=np.zeros(n_sb - 1),
                   ray_theta=np.zeros(n_rays), ray_phi=np.zeros(n_rays), ray_domega=np.zeros(n_rays))
        rc = self.lib.b200rt_make_grid_sph(self.precision, n_rb, n_sb, n_theta, n_phi, out["radial_boundaries"],
                                           szamethod, raymethod, out["sza_boundaries"], out["pts_radii"],
                                           out["pts_sza"], out["ray_theta"], out["ray_phi"], out["ray_domega"])
        if rc != 0:
            raise B200RTError(f"b200rt_make_grid_sph: status {rc}")
        return out

    def set_grid(self, g):
        n_rb, n_sb, n_rays = len(g["radial_boundaries"]), len(g["sza_boundaries"]), len(g["ray_theta"])
        self._ck(self.lib.b200rt_set_grid_sph(self.h, n_rb, n_sb, n_rays, g["radial_boundaries"], g["sza_boundaries"],
                                              g["pts_radii"], g["pts_sza"], g["ray_theta"], g["ray_phi"],
                                              g["ray_domega"]))
        self.n_rb, self.n_sb, self.n_rays = n_rb, n_sb, n_rays
        self.n_vox = (n_rb - 1) * (n_sb - 1)
        self.cap = 2 * n_rb + n_sb

    def make_grid_pp(self, n_rb, n_theta, rb):
        """plane_parallel_grid<n_rb, n_theta>::setup_voxels / setup_rays"""
        out = dict(radial_boundaries=np.ascontiguousarray(rb, dtype=np.float64), pts_radii=np.zeros(n_rb - 1),
                   ray_theta=np.zeros(n_theta), ray_domega=np.zeros(n_theta))
        rc = self.lib.b200rt_make_grid_pp(self.precision, n_rb, n_theta, out["radial_boundaries"], out["pts_radii"],
                                          out["ray_theta"], out["ray_domega"])
        if rc != 0:
            raise B200RTError(f"b200rt_make_grid_pp: status {rc}")
        return out

    def set_grid_pp(self, g):
        n_rb, n_rays = len(g["radial_boundaries"]), len(g["ray_theta"])
        self._ck(self.lib.b200rt_set_grid_pp(self.h, n_rb, n_rays, g["radial_boundaries"], g["pts_radii"],
                                             g["ray_theta"], g["ray_domega"]))
        self.n_rb, self.n_sb, self.n_rays = n_rb, 2, n_rays
        self.n_vox = n_rb - 1
        self.cap = 2 * n_rb + 2

    # ---- emissions
    def set_singlet(self, e, n_em, branching, T_ref, sigma_ref, g, tabs):
        self.mult = None
        """tabs: dict with the eight per-voxel tables of singlet_CFR (names as in the reference)"""
        names = ("T_ratio", "density", "dtau_species", "dtau_absorber",
                 "T_ratio_pt", "density_pt", "dtau_species_pt", "dtau_absorber_pt")
        arrs = [np.ascontiguousarray(tabs[k], dtype=np.float64) for k in names]
        self._ck(self.lib.b200rt_set_singlet(self.h, e, n_em, branching, T_ref, sigma_ref, g, *arrs))
        self.n_em = n_em

    def multiplet_desc(self, kind, solar):
        """tracker constants of the reference for `kind` + the pumping fluxes: O I: solar[0] = Lyman beta flux on
        every line; H: solar[0] on the Lyman alpha lines, solar[1] on the Lyman beta lines"""
        load()
        d = MultipletDesc()
        rc = self.lib.b200rt_multiplet_desc_init(kind, self.precision, C.byref(d))
        if rc != 0:
            raise B200RTError(f"b200rt_multiplet_desc_init: status {rc}")
        for l in range(d.n_lines):
            d.solar_flux[l] = float(solar[0]) if (kind == 0 or d.multiplet_index[l] == 0) else float(solar[1])
        return d

    def set_multiplet(self, desc, tabs):
        """tabs: species_density[_pt] [n_lower][n_vox], species_T[_pt], absorber_density[_pt] [n_vox]"""
        names = ("species_density", "species_density_pt", "species_T", "species_T_pt", "absorber_density",
                 "absorber_density_pt")
        arrs = [np.ascontiguousarray(tabs[k], dtype=np.float64).ravel() for k in names]
        self._ck(self.lib.b200rt_set_multiplet(self.h, C.byref(desc), *arrs))
        self.mult = desc
        self.n_em = 1

    # ---- source function
    def generate_S(self):
        self._ck(self.lib.b200rt_generate_S(self.h))

    def influence(self, v_begin=0, v_end=None):
        self._ck(self.lib.b200rt_influence(self.h, v_begin, self.n_vox if v_end is None else v_end))

    def solve(self):
        self._ck(self.lib.b200rt_solve(self.h))

    def last_step_count(self):
        n = C.c_longlong(0)
        self._ck(self.lib.b200rt_last_step_count(self.h, C.byref(n)))
        return n.value

    def last_substep_count(self):
        n = C.c_longlong(0)
        self._ck(self.lib.b200rt_last_substep_count(self.h, C.byref(n)))
        return n.value

    def solution(self, e, want_S=True):
        m = getattr(self, "mult", None)
        n_el = self.n_vox * (m.n_upper if m else 1)
        n_ln = self.n_vox * (m.n_lines if m else 1)
        S = np.zeros(n_el) if want_S else None
        S0, tsp, tab = np.zeros(n_el), np.zeros(n_ln), np.zeros(n_ln)
        self._ck(self.lib.b200rt_get_solution(self.h, e, _ptr(S), _ptr(S0), _ptr(tsp), _ptr(tab)))
        return dict(S=S, S0=S0, tau_species_ss=tsp, tau_absorber_ss=tab)

    def influence_matrix(self, e, layout=ROW_MAJOR):
        m = getattr(self, "mult", None)
        n_el = self.n_vox * (m.n_upper if m else 1)
        K = np.zeros((n_el, n_el))
        self._ck(self.lib.b200rt_get_influence(self.h, e, layout, K))
        return K

    def set_sourcefn(self, e, S):
        self._ck(self.lib.b200rt_set_sourcefn(self.h, e, np.ascontiguousarray(S, dtype=np.float64)))

    def residual(self, e):
        r = C.c_double(0)
        self._ck(self.lib.b200rt_last_residual(self.h, e, C.byref(r)))
        return r.value

    def influence_dev(self, e):
        p = [_vp() for _ in range(4)]
        self._ck(self.lib.b200rt_influence_dev(self.h, e, *[C.byref(x) for x in p]))
        return [x.value for x in p]

    def influence_ranges(self, ranges):
        """ranges: [(v_begin, v_end), ...] ascending and disjoint (multi.partition_interleaved)"""
        a = np.ascontiguousarray([r[0] for r in ranges], dtype=np.int32)
        b = np.ascontiguousarray([r[1] for r in ranges], dtype=np.int32)
        self._ck(self.lib.b200rt_influence_ranges(self.h, len(a), a, b))

    # ---- multi-GPU row exchange over peer memory (include/b200rt.h)
    def ipc_export_influence(self, e=0) -> bytes:
        buf = C.create_string_buffer(64)
        self._ck(self.lib.b200rt_ipc_export_influence(self.h, e, buf))
        return buf.raw

    def ipc_open(self, handle: bytes) -> int:
        p = C.c_void_p()
        self._ck(self.lib.b200rt_ipc_open(self.h, handle, C.byref(p)))
        return p.value

    def ipc_close(self, ptr):
        self._ck(self.lib.b200rt_ipc_close(self.h, ptr))

    def set_row_sink(self, e, ptr):
        self._ck(self.lib.b200rt_set_row_sink(self.h, e, ptr))

    # ---- distributed solve (include/b200rt.h): the rows stay where they were built
    def solve_exchange(self, want_ipc=False):
        """-> (device pointer of this context's exchange block, its 64-byte CUDA IPC handle or None)"""
        p = C.c_void_p()
        buf = C.create_string_buffer(64) if want_ipc else None
        self._ck(self.lib.b200rt_solve_exchange(self.h, C.byref(p), buf))
        return p.value, (buf.raw if want_ipc else None)

    def solve_distributed(self, rank, world, blocks):
        """blocks[q]: rank q's exchange block as addressable from this process (blocks[rank]: the own one)"""
        arr = (C.c_void_p * world)(*[C.c_void_p(b) for b in blocks])
        self._ck(self.lib.b200rt_solve_distributed(self.h, rank, world, arr))

    def last_solve_steps(self):
        n = C.c_int(0)
        self._ck(self.lib.b200rt_last_solve_steps(self.h, C.byref(n)))
        return n.value

    # ---- observations
    def los_from_MSO(self, locs, dirs):
        n = len(locs)
        out = [np.zeros(n) for _ in range(9)]
        rc = self.lib.b200rt_los_from_MSO(self.precision, n, np.ascontiguousarray(locs, dtype=np.float64),
                                          np.ascontiguousarray(dirs, dtype=np.float64), *out)
        if rc != 0:
            raise B200RTError(f"b200rt_los_from_MSO: status {rc}")
        return out

    def brightness(self, los, n_subsamples=10, out=None):
        """host buffers in, host buffers out: the reference-facing call (brightness_gpu).  `out`: four caller-owned
        float64 arrays of shape (rows, n) to receive the results (e.g. page-locked buffers that are re-used)."""
        n = len(los[0])
        if out is None:
            out = [np.zeros((r, n)) for r in self._out_rows()]
        self._ck(self.lib.b200rt_brightness(self.h, n, *los, n_subsamples, *[_ptr(o) for o in out]))
        self.n_los = n
        return dict(brightness=out[0], tau_species_final=out[1], tau_absorber_final=out[2], species_col_dens=out[3])

    def los_upload(self, los):
        self.n_los = len(los[0])
        self._ck(self.lib.b200rt_los_upload(self.h, self.n_los, *los))

    def brightness_resident(self, n_subsamples=10):
        self._ck(self.lib.b200rt_brightness_resident(self.h, n_subsamples))

    def _out_rows(self):
        m = getattr(self, "mult", None)
        return (m.n_lines, m.n_lines, m.n_lines, m.n_lower) if m else (self.n_em,) * 4

    def los_download(self):
        out = [np.zeros((r, self.n_los)) for r in self._out_rows()]
        self._ck(self.lib.b200rt_los_download(self.h, *[_ptr(o) for o in out]))
        return dict(brightness=out[0], tau_species_final=out[1], tau_absorber_final=out[2], species_col_dens=out[3])

    # ---- interplanetary hydrogen background
    def iph_load_table(self, fname):
        self._ck(self.lib.b200rt_iph_load_table(self.h, os.fsencode(fname)))

    def iph_set_table(self, tab):
        """tab: dict with kmax, lmax, ninf, temp, alt_au, ang, dans, sot, so, sn, dinf_cm3 (file layout)"""
        f = lambda k: np.ascontiguousarray(tab[k], dtype=np.float32)
        self._ck(self.lib.b200rt_iph_set_table(self.h, int(tab["kmax"]), int(tab["lmax"]), int(tab["ninf"]),
                                               float(tab["temp"]), f("alt_au"), f("ang"), f("dans"), f("sot"), f("so"),
                                               f("sn"), f("dinf_cm3")))

    def iph_background(self, fs, pos, u, v, w, want_steps=False):
        n = len(u)
        fln = np.zeros(n, np.float32)
        steps = np.zeros(n, np.int32) if want_steps else None
        a = [np.ascontiguousarray(x, dtype=np.float32) for x in (u, v, w)]
        self._ck(self.lib.b200rt_iph_background(self.h, fs, pos[0], pos[1], pos[2], n, *a, fln, _ptr(steps)))
        return (fln, steps) if want_steps else fln

    def iph_model(self, g_lya, marspos, ra, dec):
        n = len(ra)
        out = np.zeros(n)
        self._ck(self.lib.b200rt_iph_model(self.h, g_lya, np.ascontiguousarray(marspos, dtype=np.float64), n,
                                           np.ascontiguousarray(ra, dtype=np.float64),
                                           np.ascontiguousarray(dec, dtype=np.float64), out))
        return out

    def iph_extinction(self, iph, tau_abs):
        iph = np.ascontiguousarray(iph, dtype=np.float64)
        tau = np.ascontiguousarray(tau_abs, dtype=np.float64)
        out = np.zeros_like(iph)
        rc = self.lib.b200rt_iph_extinction(iph.size, iph.ravel(), tau.ravel(), out.ravel())
        if rc != 0:
            raise B200RTError(f"b200rt_iph_extinction: status {rc}")
        return out

    # ---- traversal (parity surface)
    def traverse_voxel_rays(self, v0=0, v1=None):
        v1 = self.n_vox if v1 is None else v1
        nr = (v1 - v0) * self.n_rays
        cap = nr * self.cap
        ln, eb = np.zeros(nr, np.int32), np.zeros(nr, np.int32)
        ent, dist = np.zeros(cap, np.int32), np.zeros(cap)
        n = C.c_longlong(0)
        self._ck(self.lib.b200rt_traverse_voxel_rays(self.h, v0, v1, cap, ln, eb, ent, dist, C.byref(n)))
        return ln, eb, ent[:n.value].copy(), dist[:n.value].copy()

    def traverse_los(self):
        cap = self.n_los * self.cap
        ln, eb = np.zeros(self.n_los, np.int32), np.zeros(self.n_los, np.int32)
        ent, dist = np.zeros(cap, np.int32), np.zeros(cap)
        n = C.c_longlong(0)
        self._ck(self.lib.b200rt_traverse_los(self.h, cap, ln, eb, ent, dist, C.byref(n)))
        return ln, eb, ent[:n.value].copy(), dist[:n.value].copy()

    # ---- timing
    def kernel_ms(self, phase):
        ms, nl = C.c_float(0), C.c_int(0)
        self._ck(self.lib.b200rt_last_kernel_ms(self.h, phase, C.byref(ms), C.byref(nl)))
        return ms.value, nl.value

    def synchronize(self):
        self._ck(self.lib.b200rt_synchronize(self.h))

    def fp64_peaks(self):
        """-> (DFMA TFLOP/s, DMMA TFLOP/s) measured on this device"""
        a, b = C.c_double(0), C.c_double(0)
        self._ck(self.lib.b200rt_measure_fp64_peaks(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value


def define_singlet_tables(scn, e, precision=F64):
    """Host restatement of singlet_CFR::define (reference emission/singlet_CFR.hpp:419-492):
    the eight per-voxel tables from the atmosphere's voxel averages / point values.
    Evaluated in the arithmetic of `precision`, left to right as the reference does."""
    rt = np.float64 if precision == F64 else np.float32
    n_avg, n_pt, T_avg, T_pt, a_avg, a_pt = (scn.vox_in[k].astype(rt) for k in range(6))
    T_ref, sigma_ref = rt(scn.em_scalars[e][1]), rt(scn.em_scalars[e][2])
    sig = rt(scn.abs_sigma[e])
    Tr, Tr_pt = T_ref / T_avg, T_ref / T_pt
    tabs = dict(T_ratio=Tr, T_ratio_pt=Tr_pt, density=n_avg, density_pt=n_pt,
                dtau_species=n_avg * sigma_ref * np.sqrt(Tr), dtau_species_pt=n_pt * sigma_ref * np.sqrt(Tr_pt),
                dtau_absorber=a_avg * sig, dtau_absorber_pt=a_pt * sig)
    return {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in tabs.items()}


class GpuModel:
    """Scenario-level convenience: one synthetic Scenario (synth.py) on one GPU, with the
    method vocabulary the parity tests use (grid / traverse / build_rows / solve / brightness)."""

    def __init__(self, scn, precision="f64", device=0, devices=None):
        self.scn = scn
        self.prec = F64 if precision == "f64" else F32
        self.ctx = Context(device, self.prec, devices=devices)
        if getattr(scn, "pp", False):
            self.g = self.ctx.make_grid_pp(scn.n_rb, scn.n_theta, scn.rb)
            self.ctx.set_grid_pp(self.g)
        else:
            self.g = self.ctx.make_grid(scn.n_rb, scn.n_sb, scn.n_theta, scn.n_phi, scn.rb, scn.szamethod, scn.raymethod)
            self.ctx.set_grid(self.g)
        self.n_vox, self.n_rays = self.ctx.n_vox, self.ctx.n_rays
        for e in range(scn.n_em):
            b, T, s, g = (float(x) for x in scn.em_scalars[e])
            self.ctx.set_singlet(e, scn.n_em, b, T, s, g, define_singlet_tables(scn, e, self.prec))

    def grid(self):
        nphi = self.scn.n_phi
        g = dict(self.g)
        if getattr(self.scn, "pp", False):
            return g
        g["ray_theta"] = self.g["ray_theta"][::nphi].copy()
        g["ray_phi"] = self.g["ray_phi"][:nphi].copy()
        return g

    def traverse_voxel_rays(self, v0=0, v1=None):
        return self.ctx.traverse_voxel_rays(v0, v1)

    def traverse_los(self, locs, dirs):
        self.ctx.los_upload(self.ctx.los_from_MSO(locs, dirs))
        return self.ctx.traverse_los()

    def build_rows(self, v0=0, v1=None):
        self.ctx.influence(v0, v1)
        return self.ctx.kernel_ms(PH_INFLUENCE)[0] * 1e-3, self.ctx.last_step_count()

    def solve(self):
        self.ctx.solve()
        return [self.ctx.residual(e) for e in range(self.scn.n_em)]

    def K(self, e):
        return self.ctx.influence_matrix(e)

    def vectors(self, e, want_S=True):
        return self.ctx.solution(e, want_S)

    def set_sourcefn(self, e, S):
        self.ctx.set_sourcefn(e, S)

    def brightness(self, locs, dirs, n_subsamples=10):
        los = self.ctx.los_from_MSO(locs, dirs)
        r = self.ctx.brightness(los, n_subsamples)
        out = np.stack([r["brightness"], r["tau_species_final"], r["tau_absorber_final"], r["species_col_dens"]], axis=1)
        return self.ctx.kernel_ms(PH_BRIGHTNESS)[0] * 1e-3, out


def define_multiplet_tables(scn, precision=F64):
    """Host restatement of O_1026_emission::define (reference emission/O_1026.hpp:134-217: Boltzmann populations of
    the three J levels of the O I ground term) and H_lyman_multiplet::define (emission/H_lyman_multiplet.hpp:160-217),
    evaluated in the arithmetic of `precision`."""
    rt = np.float64 if precision == F64 else np.float32
    n_avg, n_pt, T_avg, T_pt, a_avg, a_pt = (scn.vox_in[k].astype(rt) for k in range(6))
    if scn.kind == 0:
        kB, erg_per_eV = rt(1.38e-16), rt(1.60218e-12)
        E = [rt(0.0281416) * erg_per_eV, rt(0.0196224) * erg_per_eV, rt(0.0) * erg_per_eV]   # O_1026_tracker.hpp:103-110
        gw = [rt(1), rt(3), rt(5)]

        def pops(T, bulk):
            fr = [gw[l] * np.exp(-E[l] / kB / T) for l in range(3)]
            tot = fr[0] + fr[1] + fr[2]
            return np.stack([(fr[l] / tot) * bulk for l in range(3)])
        dens, dens_pt = pops(T_avg, n_avg), pops(T_pt, n_pt)
    else:
        dens, dens_pt = n_avg[None, :], n_pt[None, :]
    tabs = dict(species_density=dens, species_density_pt=dens_pt, species_T=T_avg, species_T_pt=T_pt,
                absorber_density=a_avg, absorber_density_pt=a_pt)
    return {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in tabs.items()}


class GpuMultiplet:
    """One MultipletScenario (synth.py) on one GPU, with the vocabulary of oracle/multbind.py."""

    def __init__(self, scn, precision="f64", device=0, devices=None):
        self.scn = scn
        self.prec = F64 if precision == "f64" else F32
        self.ctx = Context(device, self.prec, devices=devices)
        self.g = self.ctx.make_grid(scn.n_rb, scn.n_sb, scn.n_theta, scn.n_phi, scn.rb, scn.szamethod, scn.raymethod)
        self.ctx.set_grid(self.g)
        self.desc = self.ctx.multiplet_desc(scn.kind, scn.solar)
        self.tabs = define_multiplet_tables(scn, self.prec)
        self.ctx.set_multiplet(self.desc, self.tabs)
        d = self.desc
        self.n_vox, self.n_rays = self.ctx.n_vox, self.ctx.n_rays
        self.n_lines, self.n_mult, self.n_lower, self.n_upper, self.n_lambda = (d.n_lines, d.n_multiplets, d.n_lower,
                                                                                  d.n_upper, d.n_lambda)
        self.n_el = self.n_vox * self.n_upper

    def constants(self):
        d, NL = self.desc, self.desc.n_lines
        a = lambda f, dt=np.float64, n=NL: np.array(list(f)[:n], dtype=dt)
        return dict(multiplet_index=a(d.multiplet_index, np.int32), lower_level_index=a(d.lower_level_index, np.int32),
                    upper_level_index=a(d.upper_level_index, np.int32), line_sigma_total=a(d.line_sigma_total),
                    line_A=a(d.line_A), absorber_xsec=a(d.absorber_xsec),
                    upper_state_decay_rate=a(d.upper_state_decay_rate, n=d.n_upper), offset=a(d.offset), norm=a(d.norm),
                    weight=a(d.weight))

    def arrays(self):
        t, out = self.tabs, {}
        for l in range(self.n_lower):
            out[f"species_density_{l}"], out[f"species_density_pt_{l}"] = t["species_density"][l], t["species_density_pt"][l]
        out.update(species_T=t["species_T"], species_T_pt=t["species_T_pt"], absorber_density=t["absorber_density"],
                   absorber_density_pt=t["absorber_density_pt"])
        return out

    def build_rows(self, v0=0, v1=None):
        self.ctx.influence(v0, v1)
        return self.ctx.kernel_ms(PH_INFLUENCE)[0] * 1e-3, self.ctx.last_step_count()

    def build_ranges(self, ranges):
        """the element rows of the source voxels in `ranges` (ascending, disjoint: multi.partition_interleaved), as one
        rank of a distributed solve holds them"""
        self.ctx.influence_ranges(ranges)
        return self.ctx.kernel_ms(PH_INFLUENCE)[0] * 1e-3, self.ctx.last_step_count()

    def solve(self):
        self.ctx.solve()
        return self.ctx.residual(0)

    def last_solve_steps(self):
        """GMRES steps of the last distributed (or GMRES-chosen) solve"""
        return self.ctx.last_solve_steps()

    def K(self):
        return self.ctx.influence_matrix(0)

    def vectors(self, want_S=True):
        r = self.ctx.solution(0, want_S)
        if r["S"] is None:
            r["S"] = np.zeros(self.n_el)
        return r

    def set_sourcefn(self, S):
        self.ctx.set_sourcefn(0, S)

    def brightness(self, locs, dirs, n_subsamples=10):
        return self.ctx.brightness(self.ctx.los_from_MSO(locs, dirs), n_subsamples)
