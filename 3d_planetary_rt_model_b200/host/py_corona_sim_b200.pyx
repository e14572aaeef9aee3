# distutils: language = c++
# py_corona_sim_b200.pyx -- the reference's Cython binding plus a buffer-protocol / nogil fast path.
#
# The first statement below includes the reference's OWN binding (python/py_corona_sim.pyx) textually, from the reference
# tree at build time (oracle/build_pyx.py puts <reference>/python on the include path; nothing is copied): every class,
# method name and argument list of the reference module is therefore present unchanged.  What follows adds
# Pyobservation_fit_b200, a subclass whose hot methods take any buffer (numpy array, memoryview, ...) as a typed
# memoryview and run WITHOUT the GIL:
#   * the reference moves lines of sight element by element through Python-level loops into vector<vector<Real>>
#     (py_corona_sim.pyx:210-220, 232-247): ~6 Python assignments per line of sight, seconds for 10^6 of them, against
#     the ~60 ms the GPU needs for the whole job;
#   * its result getters go through a Python list of lists (np.asarray(vector<vector<Real>>), :460-476).
# Here both directions are one memcpy-speed pass, and generate_source_function* / brightness release the GIL, so several
# Python threads can drive several observation_fit objects (several GPUs) at once.
include "py_corona_sim.pyx"

cdef extern from "fast_binding.hpp" namespace "b200_fast" nogil:
    void b200_add_observation "b200_fast::add_observation"(observation_fit *o, const double *loc, const double *dir, int n) except +
    void b200_add_observation_ra_dec "b200_fast::add_observation_ra_dec"(observation_fit *o, const double *marspos, const double *ra, const double *dec, int n) except +
    void b200_generate_source_function "b200_fast::generate_source_function"(observation_fit *o, int kind, double nH, double x, const string &a, const string &s, bool pp, bool d) except +
    int b200_n_obs "b200_fast::n_obs"(const observation_fit *o)
    int b200_fetch "b200_fast::fetch"(observation_fit *o, int which, double *out) except +
    int b200_fetch_cols "b200_fast::fetch_cols"(observation_fit *o, int which)
    cppclass b200_csr "observation_fit::csr_matrix":
        pass
    b200_csr *b200_weights "b200_fast::weights"(observation_fit *o, int e, int which) except +
    long long b200_weights_nnz "b200_fast::weights_nnz"(const b200_csr *w)
    int b200_weights_rows "b200_fast::weights_rows"(const b200_csr *w)
    int b200_weights_cols "b200_fast::weights_cols"(const b200_csr *w)
    void b200_weights_copy "b200_fast::weights_copy"(const b200_csr *w, long long *indptr, int *indices, double *data)
    void b200_weights_free "b200_fast::weights_free"(b200_csr *w)
    cppclass b200_dvec "std::vector<double>":
        pass
    b200_dvec *b200_source_sensitivity "b200_fast::source_sensitivity"(observation_fit *o, int e, const double *w, int n, int which) except +
    int b200_vector_size "b200_fast::vector_size"(const b200_dvec *v)
    void b200_vector_copy "b200_fast::vector_copy"(const b200_dvec *v, double *out)
    void b200_vector_free "b200_fast::vector_free"(b200_dvec *v)


cdef class Pyobservation_fit_b200(Pyobservation_fit):
    """Pyobservation_fit with buffer-protocol ingest and GIL-free calls; results are identical to the base class."""

    def add_observation(self, loc_arr, dir_arr):
        cdef double[:, ::1] L = np.ascontiguousarray(loc_arr, dtype=np.float64)
        cdef double[:, ::1] D = np.ascontiguousarray(dir_arr, dtype=np.float64)
        if L.shape[0] != D.shape[0] or L.shape[1] != 3 or D.shape[1] != 3:
            raise ValueError("location and look direction must both be [n, 3]")
        cdef int n = <int> L.shape[0]
        if n == 0:
            raise ValueError("there must be at least one observation to simulate")
        with nogil:
            b200_add_observation(self.thisptr, &L[0, 0], &D[0, 0], n)

    def add_observation_ra_dec(self, mars_ecliptic_coords_arr, RA_arr, Dec_arr):
        cdef double[::1] M = np.ascontiguousarray(mars_ecliptic_coords_arr, dtype=np.float64)
        cdef double[::1] RA = np.ascontiguousarray(RA_arr, dtype=np.float64)
        cdef double[::1] DE = np.ascontiguousarray(Dec_arr, dtype=np.float64)
        if M.shape[0] != 3 or RA.shape[0] != DE.shape[0] or RA.shape[0] == 0:
            raise ValueError("mars position must be a 3-vector; RA and Dec must have the same, non-zero, length")
        cdef int n = <int> RA.shape[0]
        with nogil:
            b200_add_observation_ra_dec(self.thisptr, &M[0], &RA[0], &DE[0], n)

    cdef _generate(self, int kind, double nH, double x, atmosphere_fname, sourcefn_fname, plane_parallel, deuterium):
        cdef string a = atmosphere_fname.encode('utf-8')
        cdef string s = sourcefn_fname.encode('utf-8')
        cdef bool pp = plane_parallel
        cdef bool d = deuterium
        with nogil:
            b200_generate_source_function(self.thisptr, kind, nH, x, a, s, pp, d)

    def generate_source_function(self, Real nH, Real T, atmosphere_fname="", sourcefn_fname="",
                                 plane_parallel=False, deuterium=False):
        self._generate(0, nH, T, atmosphere_fname, sourcefn_fname, plane_parallel, deuterium)

    def generate_source_function_lc(self, Real nH, Real lc, atmosphere_fname="", sourcefn_fname="",
                                    plane_parallel=False, deuterium=False):
        self._generate(1, nH, lc, atmosphere_fname, sourcefn_fname, plane_parallel, deuterium)

    def generate_source_function_effv(self, Real nH, Real effv, atmosphere_fname="", sourcefn_fname="",
                                      plane_parallel=False, deuterium=False):
        self._generate(2, nH, effv, atmosphere_fname, sourcefn_fname, plane_parallel, deuterium)

    cdef _fetch(self, int which):
        cdef int rows
        cdef int cols = b200_fetch_cols(self.thisptr, which)
        cdef int n_rows = 2                                                       # every getter is [n_emissions][n_obs]
        out = np.empty((max(n_rows, 1), max(cols, 1)), dtype=np.float64)
        cdef double[:, ::1] O = out
        with nogil:
            rows = b200_fetch(self.thisptr, which, &O[0, 0])   # the device work of brightness() happens here, GIL released
        return out[:rows, :cols]

    def brightness(self):
        return self._fetch(0)

    def species_col_dens(self):
        return self._fetch(1)

    def tau_species_final(self):
        return self._fetch(2)

    def tau_absorber_final(self):
        return self._fetch(3)

    def iph_brightness_observed(self):
        return self._fetch(4)

    def iph_brightness_unextincted(self):
        return self._fetch(5)

    def D_brightness(self):
        return self._fetch(6)

    def D_col_dens(self):
        return self._fetch(7)

    def tau_D_final(self):
        return self._fetch(8)

    def brightness_weights(self, int i_emission, int which=0):
        """line-of-sight weighting functions of the H (which = 0) or D (1) model for the current observations:
        (indptr, indices, data) with scipy.sparse.csr_matrix((data, indices, indptr), shape=(n_obs, n_voxels)) times
        the source function = the brightness without the IPH term"""
        cdef b200_csr *w
        with nogil:
            w = b200_weights(self.thisptr, i_emission, which)
        cdef long long nnz = b200_weights_nnz(w)
        indptr = np.empty(b200_weights_rows(w) + 1, dtype=np.int64)
        indices = np.empty(max(nnz, 1), dtype=np.int32)
        data = np.empty(max(nnz, 1), dtype=np.float64)
        cdef long long[::1] P = indptr
        cdef int[::1] I = indices
        cdef double[::1] D = data
        b200_weights_copy(w, &P[0], &I[0], &D[0])
        b200_weights_free(w)
        return indptr, indices[:nnz], data[:nnz]

    def brightness_source_sensitivity(self, int i_emission, obs_weights, int which=0):
        """d(sum_l obs_weights[l] * brightness_l) / dS0 over the voxels of the H (which = 0) or D (1) model: one
        adjoint solve on the model's influence matrix (the IPH term does not depend on S0)"""
        cdef double[::1] W = np.ascontiguousarray(obs_weights, dtype=np.float64)
        cdef int n = W.shape[0]
        cdef const double *wp = &W[0] if n > 0 else NULL
        cdef b200_dvec *v
        with nogil:
            v = b200_source_sensitivity(self.thisptr, i_emission, wp, n, which)
        out = np.empty(max(b200_vector_size(v), 1), dtype=np.float64)
        cdef double[::1] O = out
        b200_vector_copy(v, &O[0])
        cdef int m = b200_vector_size(v)
        b200_vector_free(v)
        return out[:m]
