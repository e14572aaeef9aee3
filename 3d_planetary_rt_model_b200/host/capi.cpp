// capi.cpp -- flat C handles over the observation_fit facade, for ctypes-driven tests and for bindings
// that cannot consume C++ (the reference's own binding is Cython on the C++ class, python/py_corona_sim.pyx).
#include <fstream>
#include <map>
#include <mutex>
#include <csignal>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <execinfo.h>
#include <unistd.h>
#include <string>
#include <vector>
#include "observation_fit.hpp"

namespace {
thread_local std::string g_err;
template <class F> int guard(F f) {
  try { f(); return 0; } catch (const std::exception &e) { g_err = e.what(); return 1; }
}
std::vector<std::vector<double>> rows3(int n, const double *a) {
  std::vector<std::vector<double>> r(n, std::vector<double>(3));
  for (int i = 0; i < n; i++) for (int k = 0; k < 3; k++) r[i][k] = a[3 * (size_t) i + k];
  return r;
}
void flatten(const std::vector<std::vector<double>> &v, double *out) {
  size_t p = 0;
  for (auto &r : v) { std::memcpy(out + p, r.data(), r.size() * sizeof(double)); p += r.size(); }
}
}

namespace {
// B200RT_HOST_BACKTRACE=1: print a native backtrace on SIGSEGV (development aid)
void segv_handler(int sig) {
  void *frames[64];
  const int n = backtrace(frames, 64);
  const char msg[] = "libb200rt_host: fatal signal, native backtrace:\n";
  (void) !write(2, msg, sizeof msg - 1);
  backtrace_symbols_fd(frames, n, 2);
  _exit(128 + sig);
}
struct install_handler {
  install_handler() { if (getenv("B200RT_HOST_BACKTRACE")) signal(SIGSEGV, segv_handler); }
} g_install_handler;
}

// obsfit_brightness_weights keeps the matrix here until obsfit_brightness_weights_get copies it out
namespace {
std::mutex g_weights_mu;
std::map<void *, observation_fit::csr_matrix> g_weights;
}

extern "C" {
const char *obsfit_last_error() { return g_err.c_str(); }
void *obsfit_create_ex(const char *iph_fname, int device, int single_precision) {
  observation_fit *o = nullptr;
  if (guard([&] { o = new observation_fit(iph_fname ? iph_fname : "", device, single_precision != 0); })) return nullptr;
  return o;
}
void *obsfit_create(const char *iph_fname, int device) {
  observation_fit *o = nullptr;
  if (guard([&] { o = new observation_fit(iph_fname ? iph_fname : "", device); })) return nullptr;
  return o;
}
void obsfit_destroy(void *h) {
  {
    std::lock_guard<std::mutex> lock(g_weights_mu);
    g_weights.erase(h);
  }
  delete static_cast<observation_fit *>(h);
}
int obsfit_add_observation(void *h, int n, const double *loc, const double *dir) {
  return guard([&] { static_cast<observation_fit *>(h)->add_observation(rows3(n, loc), rows3(n, dir)); });
}
int obsfit_set_g_factor(void *h, double g_lya, double g_lyb) {
  return guard([&] { std::vector<double> g = {g_lya, g_lyb}; static_cast<observation_fit *>(h)->set_g_factor(g); });
}
int obsfit_add_observation_ra_dec(void *h, const double *marspos, int n, const double *ra, const double *dec) {
  return guard([&] {
    static_cast<observation_fit *>(h)->add_observation_ra_dec(std::vector<double>(marspos, marspos + 3),
                                                              std::vector<double>(ra, ra + n), std::vector<double>(dec, dec + n));
  });
}
int obsfit_generate_source_function(void *h, double nH, double T, const char *sourcefn_fname) {
  return guard([&] { static_cast<observation_fit *>(h)->generate_source_function(nH, T, "", sourcefn_fname ? sourcefn_fname : ""); });
}
int obsfit_set_use_CO2_absorption(void *h, int use) { return guard([&] { static_cast<observation_fit *>(h)->set_use_CO2_absorption(use != 0); }); }
int obsfit_set_CO2_exobase_density(void *h, double n) { return guard([&] { static_cast<observation_fit *>(h)->set_CO2_exobase_density(n); }); }
int obsfit_save_influence_matrix(void *h, const char *fname) { return guard([&] { static_cast<observation_fit *>(h)->save_influence_matrix(fname); }); }
// which: 0 brightness, 1 species_col_dens, 2 tau_species_final, 3 tau_absorber_final, 4 iph observed, 5 iph unextincted
// [2][n_obs];  6 D_brightness, 7 D_col_dens, 8 tau_D_final [2][n_obs];  9 O_1026_brightness [6][n_obs];
// 10 lyman_multiplet_brightness, 11 lyman_singlet_brightness [2][n_obs]
int obsfit_get(void *h, int which, double *out) {
  return guard([&] {
    auto *o = static_cast<observation_fit *>(h);
    switch (which) {
      case 0: flatten(o->brightness(), out); break;
      case 1: flatten(o->species_col_dens(), out); break;
      case 2: flatten(o->tau_species_final(), out); break;
      case 3: flatten(o->tau_absorber_final(), out); break;
      case 4: flatten(o->iph_brightness_observed(), out); break;
      case 5: flatten(o->iph_brightness_unextincted(), out); break;
      case 6: flatten(o->D_brightness(), out); break;
      case 7: flatten(o->D_col_dens(), out); break;
      case 8: flatten(o->tau_D_final(), out); break;
      case 9: flatten(o->O_1026_brightness(), out); break;
      case 10: flatten(o->lyman_multiplet_brightness(), out); break;
      case 11: flatten(o->lyman_singlet_brightness(), out); break;
      default: throw std::invalid_argument("obsfit_get: unknown quantity");
    }
  });
}
// ---- the other generate_source_function* members (names as observation_fit's)
static std::string str(const char *p) { return p ? p : ""; }
int obsfit_generate_source_function_ex(void *h, double nH, double T, const char *atmosphere_fname, const char *sourcefn_fname,
                                       int plane_parallel, int deuterium) {
  return guard([&] { static_cast<observation_fit *>(h)->generate_source_function(nH, T, str(atmosphere_fname), str(sourcefn_fname), plane_parallel != 0, deuterium != 0); });
}
int obsfit_generate_source_function_lc(void *h, double nH, double lc, int plane_parallel, int deuterium) {
  return guard([&] { static_cast<observation_fit *>(h)->generate_source_function_lc(nH, lc, "", "", plane_parallel != 0, deuterium != 0); });
}
int obsfit_generate_source_function_effv(void *h, double nH, double effv, int plane_parallel, int deuterium) {
  return guard([&] { static_cast<observation_fit *>(h)->generate_source_function_effv(nH, effv, "", "", plane_parallel != 0, deuterium != 0); });
}
int obsfit_generate_source_function_variable_thermosphere(void *h, double nH, double T, double nCO2rmin, double rexo, double rmin,
                                                          double rmax, double rmindiffusion, double T_tropo, double r_tropo,
                                                          double shape_parameter, int plane_parallel, int deuterium) {
  return guard([&] {
    static_cast<observation_fit *>(h)->generate_source_function_variable_thermosphere(nH, T, nCO2rmin, rexo, rmin, rmax, rmindiffusion, T_tropo,
                                                                                      r_tropo, shape_parameter, "", "", plane_parallel != 0,
                                                                                      deuterium != 0);
  });
}
int obsfit_generate_source_function_nH_asym(void *h, double nH, double T, double asym, int deuterium) {
  return guard([&] { static_cast<observation_fit *>(h)->generate_source_function_nH_asym(nH, T, asym, "", deuterium != 0); });
}
int obsfit_generate_source_function_temp_asym(void *h, double nHavg, double Tnoon, double Tmidnight, int deuterium) {
  return guard([&] { static_cast<observation_fit *>(h)->generate_source_function_temp_asym(nHavg, Tnoon, Tmidnight, "", deuterium != 0); });
}
int obsfit_generate_source_function_tabular_atmosphere(void *h, double rmin, double rexo, double rmax, int n_nH, const double *alt_nH,
                                                       const double *log_nH, int n_nCO2, const double *alt_nCO2, const double *log_nCO2,
                                                       int n_T, const double *alt_T, const double *T, int compute_exosphere,
                                                       int plane_parallel, int deuterium) {
  return guard([&] {
    typedef std::vector<double> V;
    static_cast<observation_fit *>(h)->generate_source_function_tabular_atmosphere(
        rmin, rexo, rmax, V(alt_nH, alt_nH + n_nH), V(log_nH, log_nH + n_nH), V(alt_nCO2, alt_nCO2 + n_nCO2), V(log_nCO2, log_nCO2 + n_nCO2),
        V(alt_T, alt_T + n_T), V(T, T + n_T), compute_exosphere != 0, plane_parallel != 0, deuterium != 0, "");
  });
}
int obsfit_O_1026_generate_source_function(void *h, double nO, double T, double solar_lyman_beta, const char *sourcefn_fname) {
  return guard([&] { static_cast<observation_fit *>(h)->O_1026_generate_source_function(nO, T, solar_lyman_beta, "", str(sourcefn_fname)); });
}
int obsfit_lyman_multiplet_generate_source_function(void *h, double nH, double T, const char *sourcefn_fname) {
  return guard([&] { static_cast<observation_fit *>(h)->lyman_multiplet_generate_source_function(nH, T, "", str(sourcefn_fname)); });
}
int obsfit_lyman_singlet_generate_source_function(void *h, double nH, double T, const char *sourcefn_fname) {
  return guard([&] { static_cast<observation_fit *>(h)->lyman_singlet_generate_source_function(nH, T, "", str(sourcefn_fname)); });
}
// the writers on plain arrays: q = [n_em][8][n_vox] in the order the file prints them (species density, species
// single-scattering tau, species cross section, absorber density, absorber tau, absorber cross section, S0, S)
int obsfit_write_S_file(const char *fname, int n_rb, int n_sb, const double *rb, const double *pts_r, const double *sb,
                        const double *pts_s, int n_em, const char *const *names, const double *q) {
  return guard([&] {
    const size_t n_vox = (size_t) (n_rb - 1) * (n_sb - 1);
    std::vector<std::vector<std::vector<double>>> Q(n_em, std::vector<std::vector<double>>(8));
    std::vector<std::string> nm;
    for (int e = 0; e < n_em; e++) {
      nm.push_back(names[e]);
      for (int k = 0; k < 8; k++) Q[e][k].assign(q + ((size_t) e * 8 + k) * n_vox, q + ((size_t) e * 8 + k + 1) * n_vox);
    }
    write_S_file(fname, false, n_rb, n_sb, std::vector<double>(rb, rb + n_rb), std::vector<double>(pts_r, pts_r + n_rb - 1),
                 std::vector<double>(sb, sb + n_sb), std::vector<double>(pts_s, pts_s + n_sb - 1), n_em, nm, Q);
  });
}
int obsfit_write_influence_file(const char *fname, int n_em, const char *const *names, const double *K, int n) {
  return guard([&] {
    std::ofstream file(fname);
    for (int e = 0; e < n_em; e++)
      write_influence(file, names[e], std::vector<double>(K + (size_t) e * n * n, K + (size_t) (e + 1) * n * n), n);
  });
}
int obsfit_save_influence_matrix_O_1026(void *h, const char *fname) { return guard([&] { static_cast<observation_fit *>(h)->save_influence_matrix_O_1026(fname); }); }
// options
int obsfit_set_use_temp_dependent_sH(void *h, int use, double constant_temp) { return guard([&] { static_cast<observation_fit *>(h)->set_use_temp_dependent_sH(use != 0, constant_temp); }); }
int obsfit_set_sza_method(void *h, int uniform_cos) {
  return guard([&] { uniform_cos ? static_cast<observation_fit *>(h)->set_sza_method_uniform_cos() : static_cast<observation_fit *>(h)->set_sza_method_uniform(); });
}
// kind 0: species density, 1: species temperature (set_H_density_tweak[_values], set_H_temp_tweak[_values])
int obsfit_set_tweak(void *h, int kind, int on, int n, const int *voxels, double factor) {
  return guard([&] {
    auto *o = static_cast<observation_fit *>(h);
    std::vector<int> v(voxels, voxels + n);
    if (kind == 0) { o->set_H_density_tweak(on != 0); o->set_H_density_tweak_values(v, factor); }
    else { o->set_H_temp_tweak(on != 0); o->set_H_temp_tweak_values(v, factor); }
  });
}
// which 0: lc_from_T, 1: eff_from_T, 2: T_from_lc, 3: T_from_eff  (observation_fit::Tconv)
int obsfit_Tconv(void *h, int which, double x, double *out) {
  return guard([&] {
    auto &t = static_cast<observation_fit *>(h)->Tconv;
    *out = which == 0 ? t.lc_from_T(x) : which == 1 ? t.eff_from_T(x) : which == 2 ? t.T_from_lc(x) : t.T_from_eff(x);
  });
}
// source function / radial boundaries of model `which` (0 H, 1 D, 2 plane-parallel H, 3 plane-parallel D)
int obsfit_source_function_ex(void *h, int e, int which, double *out) {
  return guard([&] { auto s = static_cast<observation_fit *>(h)->source_function(e, which); std::memcpy(out, s.data(), s.size() * sizeof(double)); });
}
int obsfit_radial_boundaries_ex(void *h, int which, double *out) {
  return guard([&] { auto s = static_cast<observation_fit *>(h)->radial_boundaries(which); std::memcpy(out, s.data(), s.size() * sizeof(double)); });
}
// model 0: O I 102.6 (n = 741*3), 1: Lyman multiplet (741*4), 2: Lyman singlet (741*2); returns the length in *n
int obsfit_multiplet_source_function(void *h, int model, double *out, int capacity, int *n) {
  return guard([&] {
    auto s = static_cast<observation_fit *>(h)->multiplet_source_function(model);
    if ((int) s.size() > capacity) throw std::invalid_argument("obsfit_multiplet_source_function: buffer too small");
    std::memcpy(out, s.data(), s.size() * sizeof(double));
    if (n) *n = (int) s.size();
  });
}
int obsfit_source_function(void *h, int e, double *out) {
  return guard([&] { auto s = static_cast<observation_fit *>(h)->source_function(e); std::memcpy(out, s.data(), s.size() * sizeof(double)); });
}
int obsfit_radial_boundaries(void *h, double *out) {
  return guard([&] { auto s = static_cast<observation_fit *>(h)->radial_boundaries(); std::memcpy(out, s.data(), s.size() * sizeof(double)); });
}
// line-of-sight weighting functions (observation_fit::brightness_weights): the CSR of emission e of model `which` is
// built and kept in the handle; *nnz, *n_rows, *n_cols tell the caller what to allocate for obsfit_brightness_weights_get
int obsfit_brightness_weights(void *h, int e, int which, long long *nnz, int *n_rows, int *n_cols) {
  return guard([&] {
    observation_fit::csr_matrix m = static_cast<observation_fit *>(h)->brightness_weights(e, which);
    std::lock_guard<std::mutex> lock(g_weights_mu);
    auto &w = g_weights[h];
    w = std::move(m);
    *nnz = (long long) w.indices.size();
    *n_rows = w.n_rows;
    *n_cols = w.n_cols;
  });
}
int obsfit_brightness_weights_get(void *h, long long *indptr, int *indices, double *data) {
  return guard([&] {
    std::lock_guard<std::mutex> lock(g_weights_mu);
    auto it = g_weights.find(h);
    if (it == g_weights.end()) throw std::runtime_error("obsfit_brightness_weights_get: call obsfit_brightness_weights first");
    const auto &w = it->second;
    std::memcpy(indptr, w.indptr.data(), w.indptr.size() * sizeof(long long));
    std::memcpy(indices, w.indices.data(), w.indices.size() * sizeof(int));
    std::memcpy(data, w.data.data(), w.data.size() * sizeof(double));
    g_weights.erase(it);
  });
}
// observation_fit::brightness_source_sensitivity: w[n_obs] -> out[n_vox] = d(sum_l w_l brightness_l) / dS0
int obsfit_brightness_source_sensitivity(void *h, int e, int which, int n_obs, const double *w, double *out) {
  return guard([&] {
    auto s = static_cast<observation_fit *>(h)->brightness_source_sensitivity(e, std::vector<double>(w, w + n_obs), which);
    std::memcpy(out, s.data(), s.size() * sizeof(double));
  });
}
// out[n_sets][2][n_obs]
int obsfit_brightness_batch(void *h, int n_sets, const double *nH, const double *T, int contexts_per_gpu, int n_gpus,
                            double *out, double *seconds) {
  return guard([&] {
    auto *o = static_cast<observation_fit *>(h);
    auto r = o->brightness_batch(std::vector<double>(nH, nH + n_sets), std::vector<double>(T, T + n_sets), contexts_per_gpu, n_gpus);
    size_t p = 0;
    for (auto &s : r) for (auto &e : s) { std::memcpy(out + p, e.data(), e.size() * sizeof(double)); p += e.size(); }
    if (seconds) *seconds = o->last_batch_seconds();
  });
}
// the atmosphere on its own (host only): [6][n_vox] tables and the radial boundaries for (nH, T)
int obsfit_atmosphere_tables(double nH, double nCO2, double T, int n_rb, int n_sb, int rmethod, double *rb_out, double *tables_out) {
  return guard([&] {
    b200rt_host::chamb_diff_1d atm(nH, nCO2, T);
    auto rb = atm.radial_boundaries(n_rb, rmethod);
    std::vector<double> t[6];
    atm.voxel_tables(rb, n_sb, t);
    std::memcpy(rb_out, rb.data(), rb.size() * sizeof(double));
    for (int q = 0; q < 6; q++) std::memcpy(tables_out + (size_t) q * t[q].size(), t[q].data(), t[q].size() * sizeof(double));
  });
}
}
