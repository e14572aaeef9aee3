// fast_binding.hpp -- free functions over observation_fit for a buffer-protocol / nogil Python binding
// (host/py_corona_sim_b200.pyx).  The reference's own binding (python/py_corona_sim.pyx:210-220, 232-247, 460-476) moves
// every line of sight through Python-level loops into vector<vector<Real>> and every result back through a list of
// lists; these take and fill flat arrays, so the binding can hold typed memoryviews and release the GIL.
#pragma once
#include <cstring>
#include <string>
#include <vector>
#include "observation_fit.hpp"

namespace b200_fast {

inline void add_observation(observation_fit *o, const double *loc, const double *dir, int n) { o->add_observation(loc, dir, n); }

inline void add_observation_ra_dec(observation_fit *o, const double *marspos, const double *ra, const double *dec, int n) {
  o->add_observation_ra_dec(std::vector<double>(marspos, marspos + 3), std::vector<double>(ra, ra + n), std::vector<double>(dec, dec + n));
}

// kind: 0 generate_source_function (T), 1 _lc (lambda_c), 2 _effv (effusion velocity)
inline void generate_source_function(observation_fit *o, int kind, double nH, double x, const std::string &atmosphere_fname,
                                     const std::string &sourcefn_fname, bool plane_parallel, bool deuterium) {
  if (kind == 0) o->generate_source_function(nH, x, atmosphere_fname, sourcefn_fname, plane_parallel, deuterium);
  else if (kind == 1) o->generate_source_function_lc(nH, x, atmosphere_fname, sourcefn_fname, plane_parallel, deuterium);
  else o->generate_source_function_effv(nH, x, atmosphere_fname, sourcefn_fname, plane_parallel, deuterium);
}

inline int n_obs(const observation_fit *o) { return o->n_obs(); }

// which: 0 brightness, 1 species_col_dens, 2 tau_species_final, 3 tau_absorber_final, 4 iph_brightness_observed,
// 5 iph_brightness_unextincted, 6 D_brightness, 7 D_col_dens, 8 tau_D_final -> rows of the result, out[rows][n_obs]
// (every getter of the reference is [n_emissions][n_obs], observation_fit.cpp:491-575; out may be null to ask for the
// row count only)
inline int fetch(observation_fit *o, int which, double *out) {
  std::vector<std::vector<double>> v;
  switch (which) {
    case 0: v = o->brightness(); break;
    case 1: v = o->species_col_dens(); break;
    case 2: v = o->tau_species_final(); break;
    case 3: v = o->tau_absorber_final(); break;
    case 4: v = o->iph_brightness_observed(); break;
    case 5: v = o->iph_brightness_unextincted(); break;
    case 6: v = o->D_brightness(); break;
    case 7: v = o->D_col_dens(); break;
    default: v = o->tau_D_final(); break;
  }
  if (out) {
    size_t p = 0;
    for (auto &r : v) { std::memcpy(out + p, r.data(), r.size() * sizeof(double)); p += r.size(); }
  }
  return (int) v.size();
}
inline int fetch_cols(observation_fit *o, int) { return o->n_obs(); }   // length of one row of fetch(which)

// observation_fit::brightness_weights into a matrix the caller keeps (new) and frees (weights_free) after copying it out
inline observation_fit::csr_matrix *weights(observation_fit *o, int e, int which) {
  return new observation_fit::csr_matrix(o->brightness_weights(e, which));
}
inline long long weights_nnz(const observation_fit::csr_matrix *w) { return (long long) w->indices.size(); }
inline int weights_rows(const observation_fit::csr_matrix *w) { return w->n_rows; }
inline int weights_cols(const observation_fit::csr_matrix *w) { return w->n_cols; }
inline void weights_copy(const observation_fit::csr_matrix *w, long long *indptr, int *indices, double *data) {
  std::memcpy(indptr, w->indptr.data(), w->indptr.size() * sizeof(long long));
  std::memcpy(indices, w->indices.data(), w->indices.size() * sizeof(int));
  std::memcpy(data, w->data.data(), w->data.size() * sizeof(double));
}
inline void weights_free(observation_fit::csr_matrix *w) { delete w; }

// observation_fit::brightness_source_sensitivity into a vector the caller keeps (new) and frees (vector_free)
inline std::vector<double> *source_sensitivity(observation_fit *o, int e, const double *w, int n, int which) {
  return new std::vector<double>(o->brightness_source_sensitivity(e, std::vector<double>(w, w + n), which));
}
inline int vector_size(const std::vector<double> *v) { return (int) v->size(); }
inline void vector_copy(const std::vector<double> *v, double *out) { std::memcpy(out, v->data(), v->size() * sizeof(double)); }
inline void vector_free(std::vector<double> *v) { delete v; }

}  // namespace b200_fast
