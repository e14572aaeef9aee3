// observation_fit.cpp -- see observation_fit.hpp
#include "observation_fit.hpp"
#include <cstdio>
#include <cstdlib>
#include <atomic>
#include <chrono>
#include <cmath>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <sstream>
#include <stdexcept>
#include <thread>
#include "../../include/b200rt.h"

using namespace b200rt_host;
using std::string;
using std::vector;

struct observation_fit::set_inputs {
  bool plane_parallel = false;
  int n_rb = 0, n_sb = 0, n_rays = 0, n_vox = 0;
  vector<double> rb, sb, pts_r, pts_s, ray_t, ray_p, ray_w;
  vector<double> vox[6];                 // n_avg, n_pt, T_avg, T_pt, nabs_avg, nabs_pt
  vector<double> tabs[n_hydrogen_emissions][8];
  double branching[n_hydrogen_emissions], T_ref[n_hydrogen_emissions], sigma_ref[n_hydrogen_emissions];
  double abs_sigma[n_hydrogen_emissions];
  // solution, filled after the solve (what save_S writes)
  vector<double> S[n_hydrogen_emissions], S0[n_hydrogen_emissions], tau_sp[n_hydrogen_emissions], tau_abs[n_hydrogen_emissions];
};

// one RT_grid<singlet_CFR, 2, grid> + observation of the reference (hydrogen_RT / deuterium_RT / *_pp)
struct observation_fit::singlet_model {
  b200rt_ctx *ctx = nullptr;
  set_inputs in;
  bool have_S = false, brightness_done = false, los_uploaded = false;
  vector<vector<Real>> out_q[4];                       // [quantity][i_emission][i_obs]
  vector<vector<Real>> iph_observed;                   // [i_obs][i_emission]
  const char *names[2] = {"H Lyman alpha", "H Lyman beta"};
};

// one RT_grid<multiplet emission, 1, grid> + observation (oxygen_RT / ly_multiplet_RT / ly_singlet_RT)
struct observation_fit::multiplet_model {
  b200rt_ctx *ctx = nullptr;
  b200rt_multiplet_desc desc;
  set_inputs grid;                                      // geometry only
  vector<double> dens, dens_pt, T, T_pt, absb, absb_pt; // species_density[n_lower][n_vox], ...
  vector<double> S, S0, tau_sp, tau_abs;
  string name;
  bool have_S = false;
};

void observation_fit::check(int rc, b200rt_ctx *c) const {
  if (rc != B200RT_OK)
    throw std::runtime_error(string("b200rt status ") + std::to_string(rc) + ": " + (c ? b200rt_last_error(c) : "no context"));
}

// device >= 0: that GPU.  device < 0 (the default): every visible GPU of this process behind one handle
// (b200rt_create_multi): generate_source_function splits the influence rows over them and brightness() the lines of
// sight, exactly the calls the reference's user makes (observation_fit.cpp:122-169,491-516).  B200RT_DEVICES="0,2,3"
// restricts the set; work too small to pay for the fan-out stays on the first device (include/b200rt.h).
b200rt_ctx *observation_fit::make_ctx() const {
  b200rt_ctx *c = nullptr;
  int rc;
  if (device >= 0) {
    rc = b200rt_create(device, precision, &c);
  } else {
    std::vector<int> ids;
    if (const char *env = getenv("B200RT_DEVICES")) {
      const char *p = env;
      while (*p) {
        char *end = nullptr;
        const long v = strtol(p, &end, 10);
        if (end == p) break;
        ids.push_back((int) v);
        p = (*end == ',') ? end + 1 : end;
      }
    }
    rc = b200rt_create_multi((int) ids.size(), ids.empty() ? nullptr : ids.data(), precision, &c);
  }
  if (rc != B200RT_OK)
    throw std::runtime_error("observation_fit: no usable CUDA device (this library has no CPU path)");
  return c;
}

observation_fit::observation_fit(const string iph_sfn_fnamee, int devicee, bool single_precision)
    : device(devicee), precision(single_precision ? B200RT_F32 : B200RT_F64), iph_sfn_fname(iph_sfn_fnamee) {
  // Real = float is the only precision the reference's own GPU module is built in (makefile:80,230; parity bar 1e-4);
  // the facade's interface stays double, the device arithmetic (traversal, march, brightness) runs in float, the solve in
  // FP64.  B200RT_FACADE_REAL=float selects it for callers that cannot pass the argument (the unchanged .pyx).
  if (const char *env = getenv("B200RT_FACADE_REAL"))
    if (string(env) == "float" || string(env) == "f32") precision = B200RT_F32;
  CO2_exobase_density = default_CO2_exobase_density;
  g_factor[0] = lyman_alpha_typical_g_factor;
  g_factor[1] = lyman_beta_typical_g_factor;
  H = new singlet_model;
  H->ctx = make_ctx();            // fails here, loudly, without a GPU
}

observation_fit::~observation_fit() {
  for (singlet_model *m : {H, D, H_pp, D_pp})
    if (m) { if (m->ctx) b200rt_destroy(m->ctx); delete m; }
  for (multiplet_model *m : {O, ly_multiplet, ly_singlet})
    if (m) { if (m->ctx) b200rt_destroy(m->ctx); delete m; }
}

observation_fit::singlet_model &observation_fit::singlet(int which) {
  singlet_model **slot = which == 0 ? &H : which == 1 ? &D : which == 2 ? &H_pp : &D_pp;
  if (!*slot) {
    *slot = new singlet_model;
    (*slot)->ctx = make_ctx();
    for (int e = 0; e < n_hydrogen_emissions; e++) b200rt_set_g_factor((*slot)->ctx, e, g_factor[e]);
  }
  return **slot;
}

void observation_fit::add_observation(const vector<vector<Real>> &MSO_locations, const vector<vector<Real>> &MSO_directions) {
  if (MSO_locations.size() != MSO_directions.size())
    throw std::invalid_argument("location and look direction must have the same length.");
  const int n = (int) MSO_locations.size();
  vector<double> loc(3 * (size_t) n), dir(3 * (size_t) n);
  for (int i = 0; i < n; i++)
    for (int k = 0; k < 3; k++) {
      loc[3 * (size_t) i + k] = MSO_locations[i].at(k);
      dir[3 * (size_t) i + k] = MSO_directions[i].at(k);
    }
  add_observation(loc.data(), dir.data(), n);
}

void observation_fit::add_observation(const double *loc, const double *dir, int n) {
  if (n < 0 || (n > 0 && (!loc || !dir))) throw std::invalid_argument("add_observation: bad arguments");
  for (auto &a : los) a.assign(n, 0.0);
  int rc = b200rt_los_from_MSO(precision, n, loc, dir, los[0].data(), los[1].data(), los[2].data(),
                               los[3].data(), los[4].data(), los[5].data(), los[6].data(), los[7].data(), los[8].data());
  if (rc != B200RT_OK) throw std::runtime_error("b200rt_los_from_MSO failed");
  for (singlet_model *m : {H, D, H_pp, D_pp})
    if (m) m->brightness_done = m->los_uploaded = false;
}

void observation_fit::simulate_iph(const bool sim_iphh) { sim_iph = sim_iphh; }

void observation_fit::add_observation_ra_dec(const vector<Real> &mars_ecliptic_coords, const vector<Real> &RAA,
                                             const vector<Real> &Decc) {
  simulate_iph(true);
  if ((int) RAA.size() != n_obs() || RAA.size() != Decc.size())
    throw std::invalid_argument("IPH coordinates must have the same dimensions as locations and directions");
  if (mars_ecliptic_coords.size() != 3) throw std::invalid_argument("mars ecliptic coords must be a 3D position.");
  mars_ecliptic_pos = mars_ecliptic_coords;
  ra = RAA;
  dec = Decc;
  iph_unextincted.assign(n_obs(), vector<Real>(n_hydrogen_emissions, 0.0));
  get_unextincted_iph();
}

void observation_fit::get_unextincted_iph() {
  if (!iph_table_loaded) {
    check(b200rt_iph_load_table(H->ctx, iph_sfn_fname.c_str()), H->ctx);
    iph_table_loaded = true;
  }
  vector<double> kR(n_obs());
  check(b200rt_iph_model(H->ctx, g_factor[0], mars_ecliptic_pos.data(), n_obs(), ra.data(), dec.data(), kR.data()), H->ctx);
  for (int i = 0; i < n_obs(); i++) {
    iph_unextincted[i][0] = kR[i];
    iph_unextincted[i][1] = g_factor[1] / g_factor[0] * kR[i];   // observation_fit.cpp:114-117
  }
  for (singlet_model *m : {H, D, H_pp, D_pp})
    if (m) m->brightness_done = false;
}

void observation_fit::set_g_factor(vector<Real> &g) {
  for (int e = 0; e < n_hydrogen_emissions; e++) g_factor[e] = g.at(e);
  for (singlet_model *m : {H, D, H_pp, D_pp})
    if (m) {
      for (int e = 0; e < n_hydrogen_emissions; e++) b200rt_set_g_factor(m->ctx, e, g_factor[e]);
      m->brightness_done = false;
    }
  std::cout << "Ly alpha solar brightness = " << g[0] / lyman_alpha_cross_section_total << std::endl;
  std::cout << "Ly beta solar brightness = " << g[1] / lyman_beta_cross_section_total << std::endl;
}

// ---- one parameter set: atmosphere -> grid -> the tables of singlet_CFR::define (singlet_CFR.hpp:419-492)
void observation_fit::build_inputs(const atmosphere_model &atm, const Real &Texo, bool plane_parallel, set_inputs &in) const {
  in.plane_parallel = plane_parallel;
  in.n_rb = n_radial_boundaries;
  if (!plane_parallel) {
    in.n_sb = n_sza_boundaries; in.n_rays = n_rays_theta * n_rays_phi;
    in.rb = atm.radial_boundaries(n_radial_boundaries, 0);                  // rmethod_altitude, observation_fit.cpp:34
    in.sb.assign(in.n_sb, 0); in.pts_r.assign(in.n_rb - 1, 0); in.pts_s.assign(in.n_sb - 1, 0);
    in.ray_t.assign(in.n_rays, 0); in.ray_p.assign(in.n_rays, 0); in.ray_w.assign(in.n_rays, 0);
    int rc = b200rt_make_grid_sph(precision, in.n_rb, in.n_sb, n_rays_theta, n_rays_phi, in.rb.data(), szamethod,
                                  1 /* raymethod_theta_uniform */, in.sb.data(), in.pts_r.data(), in.pts_s.data(),
                                  in.ray_t.data(), in.ray_p.data(), in.ray_w.data());
    if (rc != B200RT_OK) throw std::runtime_error("b200rt_make_grid_sph failed");
  } else {
    in.n_sb = 2; in.n_rays = n_rays_pp;
    in.rb = atm.radial_boundaries(n_radial_boundaries, 1);                  // rmethod_log_n_species, observation_fit.cpp:30-31
    in.sb = {0.0, pi}; in.pts_s = {0.0};
    in.pts_r.assign(in.n_rb - 1, 0);
    in.ray_t.assign(in.n_rays, 0); in.ray_p.assign(in.n_rays, 0); in.ray_w.assign(in.n_rays, 0);
    int rc = b200rt_make_grid_pp(precision, in.n_rb, n_rays_pp, in.rb.data(), in.pts_r.data(), in.ray_t.data(), in.ray_w.data());
    if (rc != B200RT_OK) throw std::runtime_error("b200rt_make_grid_pp failed");
  }
  in.n_vox = (in.n_rb - 1) * (in.n_sb - 1);
  atm.voxel_tables(in.rb, in.pts_r, in.sb, in.pts_s, in.vox);
  const double br[2] = {1.0, lyman_beta_branching_ratio};
  const double sref[2] = {atm.sH_lya(Texo), atm.sH_lyb(Texo)};
  for (int e = 0; e < n_hydrogen_emissions; e++) {
    in.branching[e] = br[e]; in.T_ref[e] = Texo; in.sigma_ref[e] = sref[e];
    for (auto &t : in.tabs[e]) t.assign(in.n_vox, 0.0);
    for (int v = 0; v < in.n_vox; v++) {
      const double n_avg = in.vox[0][v], n_pt = in.vox[1][v], T_avg = in.vox[2][v], T_pt = in.vox[3][v];
      const double a_avg = in.vox[4][v], a_pt = in.vox[5][v];
      const double Tr = Texo / T_avg, Tr_pt = Texo / T_pt;
      const double sa = (e == 0) ? atm.sCO2_lya(T_avg) : atm.sCO2_lyb(T_avg);
      const double sa_pt = (e == 0) ? atm.sCO2_lya(T_pt) : atm.sCO2_lyb(T_pt);
      in.abs_sigma[e] = sa;
      in.tabs[e][0][v] = Tr;                             // species_T_ratio
      in.tabs[e][1][v] = n_avg;                          // species_density
      in.tabs[e][2][v] = n_avg * sref[e] * std::sqrt(Tr);         // dtau_species
      in.tabs[e][3][v] = a_avg * sa;                     // dtau_absorber
      in.tabs[e][4][v] = Tr_pt;
      in.tabs[e][5][v] = n_pt;
      in.tabs[e][6][v] = n_pt * sref[e] * std::sqrt(Tr_pt);
      in.tabs[e][7][v] = a_pt * sa_pt;
    }
    // singlet_CFR::tweak_species_density / tweak_species_temp (singlet_CFR.hpp:494-517); `abs` = dtau_absorber /
    // dtau_species is formed on the device from the two tables, so it follows
    if (tweak_H_density)
      for (int v : tweak_H_density_voxel_numbers) {
        if (v < 0 || v >= in.n_vox) throw std::out_of_range("tweak voxel number outside the grid");
        for (int q : {1, 2, 5, 6}) in.tabs[e][q][v] *= tweak_H_density_factor;
      }
    if (tweak_H_temp)
      for (int v : tweak_H_temp_voxel_numbers) {
        if (v < 0 || v >= in.n_vox) throw std::out_of_range("tweak voxel number outside the grid");
        for (int q : {0, 4}) in.tabs[e][q][v] /= tweak_H_temp_factor;
        for (int q : {2, 6}) in.tabs[e][q][v] /= std::sqrt(tweak_H_temp_factor);
      }
  }
}

void observation_fit::load_inputs(b200rt_ctx *c, const set_inputs &in) const {
  if (in.plane_parallel)
    check(b200rt_set_grid_pp(c, in.n_rb, in.n_rays, in.rb.data(), in.pts_r.data(), in.ray_t.data(), in.ray_w.data()), c);
  else
    check(b200rt_set_grid_sph(c, in.n_rb, in.n_sb, in.n_rays, in.rb.data(), in.sb.data(), in.pts_r.data(), in.pts_s.data(),
                              in.ray_t.data(), in.ray_p.data(), in.ray_w.data()), c);
  for (int e = 0; e < n_hydrogen_emissions; e++)
    check(b200rt_set_singlet(c, e, n_hydrogen_emissions, in.branching[e], in.T_ref[e], in.sigma_ref[e], g_factor[e],
                             in.tabs[e][0].data(), in.tabs[e][1].data(), in.tabs[e][2].data(), in.tabs[e][3].data(),
                             in.tabs[e][4].data(), in.tabs[e][5].data(), in.tabs[e][6].data(), in.tabs[e][7].data()), c);
}

// generate_source_function_sph_azi_sym / _plane_parallel (observation_fit.hpp:189-294)
void observation_fit::generate(atmosphere_model &atm, const Real &Texo, bool plane_parallel, bool deuterium,
                               const string &atmosphere_fname, const string &sourcefn_fname) {
  atm.copy_H_options(H_cross_section_options);
  if (atmosphere_fname != "") atm.save(atmosphere_fname);
  singlet_model &m = singlet((plane_parallel ? 2 : 0) + (deuterium ? 1 : 0));
  const bool was_spherical = atm.spherical;
  atm.spherical = !plane_parallel;
  build_inputs(atm, Texo, plane_parallel, m.in);
  atm.spherical = was_spherical;
  load_inputs(m.ctx, m.in);
  check(b200rt_generate_S(m.ctx), m.ctx);            // RT_obj.generate_S_gpu(), observation_fit.hpp:286-290
  for (int e = 0; e < n_hydrogen_emissions; e++) {
    for (auto *v : {&m.in.S[e], &m.in.S0[e], &m.in.tau_sp[e], &m.in.tau_abs[e]}) v->assign(m.in.n_vox, 0.0);
    check(b200rt_get_solution(m.ctx, e, m.in.S[e].data(), m.in.S0[e].data(), m.in.tau_sp[e].data(), m.in.tau_abs[e].data()), m.ctx);
  }
  m.have_S = true;
  m.brightness_done = false;
  if (sourcefn_fname != "") save_S(sourcefn_fname, m.in);
}

void observation_fit::generate_source_function(const Real &nHexo, const Real &Texo, const string atmosphere_fname,
                                               const string sourcefn_fname, const bool plane_parallel, const bool deuterium) {
  chamb_diff_1d atm(rMars + 80e5, rexo_typical, 10.0, rMars + 80e5, nHexo, CO2_exobase_density, krasnopolsky_temperature(Texo),
                    deuterium ? species_density_parameters::deuterium() : species_density_parameters::hydrogen());
  generate(atm, Texo, plane_parallel, deuterium, atmosphere_fname, sourcefn_fname);
}

void observation_fit::generate_source_function_effv(const Real &nHexo, const Real &effv_exo, const string atmosphere_fname,
                                                    const string sourcefn_fname, const bool plane_parallel, const bool deuterium) {
  generate_source_function(nHexo, Tconv.T_from_eff(effv_exo), atmosphere_fname, sourcefn_fname, plane_parallel, deuterium);
}

void observation_fit::generate_source_function_lc(const Real &nHexo, const Real &lc_exo, const string atmosphere_fname,
                                                  const string sourcefn_fname, const bool plane_parallel, const bool deuterium) {
  generate_source_function(nHexo, Tconv.T_from_lc(lc_exo), atmosphere_fname, sourcefn_fname, plane_parallel, deuterium);
}

void observation_fit::generate_source_function_variable_thermosphere(const Real &nHexo, const Real &Texo, const Real &nCO2rminn,
                                                                     const Real rexoo, const Real rminn, const Real rmaxx,
                                                                     const Real rmindiffusionn, const Real T_tropo,
                                                                     const Real r_tropo, const Real shape_parameter,
                                                                     const string atmosphere_fname, const string sourcefn_fname,
                                                                     const bool plane_parallel, const bool deuterium) {
  chamb_diff_1d atm(rminn, rexoo, rmaxx, rmindiffusionn, nHexo, nCO2rminn,
                    krasnopolsky_temperature(Texo, T_tropo, r_tropo, shape_parameter, false),
                    deuterium ? species_density_parameters::deuterium() : species_density_parameters::hydrogen(),
                    chamb_diff_1d::method_rmax_nCO2rmin);
  generate(atm, Texo, plane_parallel, deuterium, atmosphere_fname, sourcefn_fname);
}

void observation_fit::generate_source_function_nH_asym(const Real &nHexo, const Real &Texo, const Real &asym,
                                                       const string sourcefn_fname, const bool deuterium) {
  // the reference builds this atmosphere with H_thermosphere whatever `deuterium` says (observation_fit.cpp:269)
  chamb_diff_1d_asymmetric atm(rMars + 80e5, rexo_typical, 10.0, rMars + 80e5, nHexo, CO2_exobase_density,
                               krasnopolsky_temperature(Texo), species_density_parameters::hydrogen());
  atm.set_asymmetry(asym);
  generate(atm, Texo, false, deuterium, "", sourcefn_fname);
}

void observation_fit::generate_source_function_temp_asym(const Real &nHavg, const Real &Tnoon, const Real &Tmidnight,
                                                         const string sourcefn_fname, const bool deuterium) {
  generate_source_function_temp_asym(nHavg, Tnoon, Tmidnight, 2.6e13, rexo_typical, rMars + 80e5, rMars + 50000e5,
                                     rMars + 80e5, 125.0, rMars + 90e5, 11.4, 2.5, sourcefn_fname, deuterium);
}

void observation_fit::generate_source_function_temp_asym(const Real &nHavg, const Real &Tnoon, const Real &Tmidnight,
                                                         const Real nCO2rminn, const Real rexoo, const Real rminn,
                                                         const Real rmaxx, const Real rmindiffusionn, const Real T_tropo,
                                                         const Real r_tropo, const Real shape_parameter, const Real Tpowerr,
                                                         const string sourcefn_fname, const bool deuterium) {
  chamb_diff_temp_asymmetric atm(species_density_parameters::hydrogen(), nHavg, Tnoon, Tmidnight, nCO2rminn, rexoo, rminn,
                                 rmaxx, rmindiffusionn, T_tropo, r_tropo, shape_parameter, Tpowerr);
  generate(atm, Tnoon, false, deuterium, "", sourcefn_fname);
}

void observation_fit::generate_source_function_tabular_atmosphere(const Real rmin, const Real rexo, const Real rmax,
                                                                  const vector<double> &alt_nH, const vector<double> &log_nH,
                                                                  const vector<double> &alt_nCO2, const vector<double> &log_nCO2,
                                                                  const vector<double> &alt_temp, const vector<double> &temp,
                                                                  const bool compute_exosphere, const bool plane_parallel,
                                                                  const bool deuterium, const string sourcefn_fname) {
  tabular_1d atm(rmin, rexo, rmax, compute_exosphere);
  atm.load_log_species_density(alt_nH, log_nH);
  atm.load_log_absorber_density(alt_nCO2, log_nCO2);
  atm.load_temperature(alt_temp, temp);
  const Real Texo = atm.Temp(rexo);
  generate(atm, Texo, plane_parallel, deuterium, "", sourcefn_fname);
}

vector<observation_fit::Real> observation_fit::source_function(int e, int which) {
  singlet_model &m = singlet(which);
  if (!m.have_S) throw std::runtime_error("observation_fit: no source function yet");
  return m.in.S[e];
}
vector<observation_fit::Real> observation_fit::radial_boundaries(int which) const {
  const singlet_model *m = which == 0 ? H : which == 1 ? D : which == 2 ? H_pp : D_pp;
  if (!m || !m->have_S) throw std::runtime_error("observation_fit: no source function yet");
  return m->in.rb;
}

// RT_grid::brightness_gpu(obs) + the packing of observation_fit.cpp:491-559
void observation_fit::run_brightness(b200rt_ctx *c, bool upload, vector<vector<Real>> (&q)[4]) const {
  const int n = n_obs();
  vector<double> flat[4];
  for (auto &f : flat) f.assign((size_t) n_hydrogen_emissions * n, 0.0);
  if (upload)
    check(b200rt_los_upload(c, n, los[0].data(), los[1].data(), los[2].data(), los[3].data(), los[4].data(),
                            los[5].data(), los[6].data(), los[7].data(), los[8].data()), c);
  check(b200rt_brightness_resident(c, 10), c);
  check(b200rt_los_download(c, flat[0].data(), flat[1].data(), flat[2].data(), flat[3].data()), c);
  for (int k = 0; k < 4; k++) {
    q[k].assign(n_hydrogen_emissions, vector<Real>());
    for (int e = 0; e < n_hydrogen_emissions; e++) q[k][e].assign(flat[k].begin() + (size_t) e * n, flat[k].begin() + (size_t) (e + 1) * n);
  }
}

void observation_fit::model_brightness(singlet_model &m) {
  if (!m.have_S) throw std::runtime_error("observation_fit: generate a source function before asking for brightness");
  if (n_obs() == 0) throw std::runtime_error("there must be at least one observation to simulate");
  if (m.brightness_done) return;
  if (sim_iph && (int) iph_unextincted.size() != n_obs())
    throw std::runtime_error("observation_fit: the IPH coordinates belong to an earlier set of observations "
                             "(call add_observation_ra_dec after add_observation, or simulate_iph(false))");
  run_brightness(m.ctx, !m.los_uploaded, m.out_q);
  m.los_uploaded = true;
  m.iph_observed.assign(n_obs(), vector<Real>(n_hydrogen_emissions, 0.0));
  if (sim_iph)                                  // observation::update_iph_extinction, observation.hpp:144-154
    for (int i = 0; i < n_obs(); i++)
      for (int e = 0; e < n_hydrogen_emissions; e++) {
        const Real ta = m.out_q[2][e][i];
        m.iph_observed[i][e] = (ta != -1) ? iph_unextincted[i][e] * std::exp(-ta) : 0.0;
      }
  m.brightness_done = true;
}

vector<vector<observation_fit::Real>> observation_fit::brightness() {
  model_brightness(*H);
  vector<vector<Real>> b = H->out_q[0];
  if (sim_iph)
    for (int e = 0; e < n_hydrogen_emissions; e++)
      for (int i = 0; i < n_obs(); i++) b[e][i] += H->iph_observed[i][e];
  return b;
}
vector<vector<observation_fit::Real>> observation_fit::species_col_dens() { model_brightness(*H); return H->out_q[3]; }
vector<vector<observation_fit::Real>> observation_fit::tau_species_final() { model_brightness(*H); return H->out_q[1]; }
vector<vector<observation_fit::Real>> observation_fit::tau_absorber_final() { model_brightness(*H); return H->out_q[2]; }
vector<vector<observation_fit::Real>> observation_fit::iph_brightness_observed() {
  model_brightness(*H);
  vector<vector<Real>> r(n_hydrogen_emissions, vector<Real>(n_obs(), 0.0));   // [i_emission][i_obs], observation_fit.cpp:561-575
  if (sim_iph)
    for (int e = 0; e < n_hydrogen_emissions; e++)
      for (int i = 0; i < n_obs(); i++) r[e][i] = H->iph_observed[i][e];
  return r;
}
vector<vector<observation_fit::Real>> observation_fit::iph_brightness_unextincted() {
  vector<vector<Real>> r(n_hydrogen_emissions, vector<Real>(n_obs(), 0.0));
  if (sim_iph)
    for (int e = 0; e < n_hydrogen_emissions; e++)
      for (int i = 0; i < n_obs(); i++) r[e][i] = iph_unextincted[i][e];
  return r;
}

observation_fit::csr_matrix observation_fit::brightness_weights(int e, int which) {
  if (which == 2 || which == 3)
    throw std::invalid_argument("brightness_weights: the plane-parallel grid has no brightness (grid_plane_parallel.hpp:304-311)");
  if (which != 0 && which != 1) throw std::invalid_argument("brightness_weights: model must be 0 (H) or 1 (D)");
  if (e < 0 || e >= n_hydrogen_emissions) throw std::invalid_argument("brightness_weights: bad emission index");
  singlet_model &m = singlet(which);
  if (!m.have_S) throw std::runtime_error("observation_fit: generate a source function before asking for brightness weights");
  if (n_obs() == 0) throw std::runtime_error("there must be at least one observation to simulate");
  b200rt_ctx *c = m.ctx;
  if (!m.los_uploaded) {
    check(b200rt_los_upload(c, n_obs(), los[0].data(), los[1].data(), los[2].data(), los[3].data(), los[4].data(),
                            los[5].data(), los[6].data(), los[7].data(), los[8].data()), c);
    m.los_uploaded = true;
  }
  long long nnz = 0;
  check(b200rt_los_weights(c, 10, &nnz), c);
  csr_matrix r;
  r.n_rows = n_obs();
  r.n_cols = m.in.n_vox;
  r.indptr.resize((size_t) r.n_rows + 1);
  r.indices.resize((size_t) nnz);
  vector<double> val((size_t) n_hydrogen_emissions * nnz);
  check(b200rt_los_weights_download(c, r.indptr.data(), r.indices.data(), val.data()), c);
  r.data.assign(val.begin() + (size_t) e * nnz, val.begin() + (size_t) (e + 1) * nnz);
  return r;
}

vector<observation_fit::Real> observation_fit::brightness_source_sensitivity(int e, const vector<Real> &obs_weights,
                                                                           int which) {
  if (which == 2 || which == 3)
    throw std::invalid_argument("brightness_source_sensitivity: the plane-parallel grid has no brightness (grid_plane_parallel.hpp:304-311)");
  if (which != 0 && which != 1) throw std::invalid_argument("brightness_source_sensitivity: model must be 0 (H) or 1 (D)");
  if (e < 0 || e >= n_hydrogen_emissions) throw std::invalid_argument("brightness_source_sensitivity: bad emission index");
  singlet_model &m = singlet(which);
  if (!m.have_S) throw std::runtime_error("observation_fit: generate a source function before asking for its sensitivity");
  if (n_obs() == 0) throw std::runtime_error("there must be at least one observation to simulate");
  if ((int) obs_weights.size() != n_obs())
    throw std::invalid_argument("brightness_source_sensitivity: one weight per observation (" + std::to_string(n_obs()) + ")");
  b200rt_ctx *c = m.ctx;
  if (!m.los_uploaded) {
    check(b200rt_los_upload(c, n_obs(), los[0].data(), los[1].data(), los[2].data(), los[3].data(), los[4].data(),
                            los[5].data(), los[6].data(), los[7].data(), los[8].data()), c);
    m.los_uploaded = true;
  }
  // W with brightness()'s n_subsamples, r = W^T w, then lambda = (I - w K)^-T r on the resident K: r . S = lambda . S0
  check(b200rt_los_weights(c, 10, nullptr), c);
  const vector<double> w(obs_weights.begin(), obs_weights.end());
  vector<double> r((size_t) m.in.n_vox), lambda((size_t) m.in.n_vox);
  check(b200rt_los_weights_apply(c, e, 1, w.data(), r.data()), c);
  check(b200rt_solve_adjoint(c, e, 1, r.data(), lambda.data(), nullptr, nullptr), c);
  return vector<Real>(lambda.begin(), lambda.end());
}

// deuterium_RT / deuterium_obs (observation_fit.cpp:591-637)
vector<vector<observation_fit::Real>> observation_fit::D_brightness() {
  singlet_model &m = singlet(1);
  model_brightness(m);
  vector<vector<Real>> b = m.out_q[0];
  if (sim_iph)
    for (int e = 0; e < n_hydrogen_emissions; e++)
      for (int i = 0; i < n_obs(); i++) b[e][i] += m.iph_observed[i][e];
  return b;
}
vector<vector<observation_fit::Real>> observation_fit::D_col_dens() { singlet_model &m = singlet(1); model_brightness(m); return m.out_q[3]; }
vector<vector<observation_fit::Real>> observation_fit::tau_D_final() { singlet_model &m = singlet(1); model_brightness(m); return m.out_q[1]; }

// ---- options (observation_fit.cpp:413-487)
void observation_fit::set_use_CO2_absorption(const bool use) {
  H_cross_section_options.no_CO2_absorption = !use;
  multiplet_CO2_absorption = use;                        // ly_multiplet / ly_singlet .set_CO2_absorption_on/off
}
void observation_fit::set_use_temp_dependent_sH(const bool use, const Real constant_temp_sH) {
  if (!use && constant_temp_sH == -1) throw std::invalid_argument("set_use_temp_dependent_sH: a constant temperature is needed");
  H_cross_section_options.temp_dependent_sH = use;
  H_cross_section_options.constant_temp_sH = constant_temp_sH;
  multiplet_constant_temp = !use;                        // set_atmosphere_temp_RT / set_constant_temp_RT
  multiplet_constant_temp_value = constant_temp_sH;
}
void observation_fit::set_sza_method_uniform() { szamethod = 0; }
void observation_fit::set_sza_method_uniform_cos() { szamethod = 1; }
void observation_fit::reset_H_lya_xsec_coef(const Real x) { H_cross_section_options.H_lya_xsec_coef = x; }
void observation_fit::reset_H_lyb_xsec_coef(const Real x) { H_cross_section_options.H_lyb_xsec_coef = x; }
void observation_fit::reset_CO2_lya_xsec(const Real x) { H_cross_section_options.CO2_lya_xsec = x; }
void observation_fit::reset_CO2_lyb_xsec(const Real x) { H_cross_section_options.CO2_lyb_xsec = x; }
observation_fit::Real observation_fit::get_CO2_exobase_density() { return CO2_exobase_density; }
void observation_fit::reset_CO2_exobase_density() { CO2_exobase_density = default_CO2_exobase_density; }
void observation_fit::set_CO2_exobase_density(const double nCO2) { CO2_exobase_density = nCO2; }
void observation_fit::set_H_density_tweak(const bool t) { tweak_H_density = t; }
void observation_fit::set_H_density_tweak_values(const vector<int> voxels, const Real f) {
  tweak_H_density_voxel_numbers = voxels;
  tweak_H_density_factor = f;
}
void observation_fit::set_H_temp_tweak(const bool t) { tweak_H_temp = t; }
void observation_fit::set_H_temp_tweak_values(const vector<int> voxels, const Real f) {
  tweak_H_temp_voxel_numbers = voxels;
  tweak_H_temp_factor = f;
}

// ---- ASCII writers (grid_spherical_azimuthally_symmetric.hpp:630-665, singlet_CFR.hpp:519-543,
// emission_voxels.hpp:235-238).  Numbers are printed the way Eigen's default IOFormat prints a
// row vector: stream precision 6, every coefficient right-aligned to the widest one, one space between.
namespace {
string row(const vector<double> &v) {
  vector<string> s(v.size());
  size_t w = 0;
  for (size_t i = 0; i < v.size(); i++) {
    std::ostringstream o;
    o << v[i];
    s[i] = o.str();
    w = std::max(w, s[i].size());
  }
  std::ostringstream o;
  for (size_t i = 0; i < v.size(); i++) {
    if (i) o << " ";
    o << std::setw((int) w) << s[i];
  }
  return o.str();
}
}

// grid.save_S + singlet_CFR::save from plain arrays (per emission: 8 arrays of n_vox, in the order the file prints them)
void write_S_file(const string &fname, bool plane_parallel, int n_rb, int n_sb, const vector<double> &rb,
                  const vector<double> &pts_r, const vector<double> &sb, const vector<double> &pts_s, int n_em,
                  const vector<string> &names, const vector<vector<vector<double>>> &q) {
  std::ofstream file(fname.c_str());
  if (!file.is_open()) return;
  file << "radial boundaries [cm]: " << row(rb) << "\n\n";
  file << "pts radii [cm]: " << row(pts_r) << "\n\n";
  if (!plane_parallel) {
    file << "sza boundaries [rad]: " << row(sb) << "\n\n";
    file << "pts sza [rad]: " << row(pts_s) << "\n\n";
  }
  const int ns = n_sb - 1, nr = n_rb - 1;
  auto slice = [&](const vector<double> &v, int j) {      // sza_slice: every voxel of SZA column j
    vector<double> r(nr);
    for (int i = 0; i < nr; i++) r[i] = v[(size_t) i * ns + j];
    return r;
  };
  static const char *labels[8] = {"Species density [cm-3]: ", "Species single scattering tau: ", "Species cross section [cm2]: ",
                                  "Absorber density [cm-3]: ", "Absorber single scattering tau: ", "Absorber cross section [cm2]: ",
                                  "Species single scattering source function S0: ", "Source function: "};
  for (int e = 0; e < n_em; e++) {
    // grid_spherical_azimuthally_symmetric.hpp:650-660 ("For <name>" + one block per SZA);
    // grid_plane_parallel.hpp:329-332 ("For <name>," + one block)
    file << "For " << names[e] << (plane_parallel ? ",\n" : "\n");
    for (int j = 0; j < ns; j++) {
      if (!plane_parallel) file << "  For SZA = " << pts_s[j] << ": \n";
      for (int k = 0; k < 8; k++) file << "    " << labels[k] << row(slice(q[e][k], j)) << (k == 7 ? "\n\n" : "\n");
    }
  }
}

void observation_fit::save_S(const string &fname, const set_inputs &in) {
  vector<vector<vector<double>>> q(n_hydrogen_emissions, vector<vector<double>>(8));
  for (int e = 0; e < n_hydrogen_emissions; e++) {
    vector<double> sig(in.n_vox), asig(in.n_vox, in.abs_sigma[e]);
    for (int v = 0; v < in.n_vox; v++) sig[v] = in.sigma_ref[e] * std::sqrt(in.tabs[e][0][v]);
    q[e] = {in.tabs[e][1], in.tau_sp[e], sig, in.vox[4], in.tau_abs[e], asig, in.S0[e], in.S[e]};
  }
  write_S_file(fname, in.plane_parallel, in.n_rb, in.n_sb, in.rb, in.pts_r, in.sb, in.pts_s, n_hydrogen_emissions,
               {"H Lyman alpha", "H Lyman beta"}, q);
}

// emission_voxels::save_influence (emission_voxels.hpp:235-238) for every emission of a model
void write_influence(std::ofstream &file, const string &name, const vector<double> &K, int n) {
  file << "Here is the influence matrix for " << name << ":\n";
  // Eigen prints a matrix with every coefficient padded to the widest one of the whole matrix
  vector<string> s(K.size());
  size_t w = 0;
  for (size_t i = 0; i < K.size(); i++) {
    std::ostringstream o;
    o << K[i];
    s[i] = o.str();
    w = std::max(w, s[i].size());
  }
  for (int r = 0; r < n; r++) {
    for (int cidx = 0; cidx < n; cidx++) {
      if (cidx) file << " ";
      file << std::setw((int) w) << s[(size_t) r * n + cidx];
    }
    file << "\n";
  }
  file << "\n";
}

void observation_fit::save_influence_matrix(const string fname) {
  if (!H->have_S) throw std::runtime_error("observation_fit: no influence matrix yet");
  std::ofstream file(fname.c_str());
  if (!file.is_open()) return;
  const int n = H->in.n_vox;
  vector<double> K((size_t) n * n);
  for (int e = 0; e < n_hydrogen_emissions; e++) {
    check(b200rt_get_influence(H->ctx, e, B200RT_ROW_MAJOR, K.data()), H->ctx);   // fetched lazily: K lives on the device
    write_influence(file, H->names[e], K, n);
  }
}

void observation_fit::save_influence_matrix_O_1026(const string fname) {
  if (!O || !O->have_S) throw std::runtime_error("observation_fit: no O 102.6 influence matrix yet");
  std::ofstream file(fname.c_str());
  if (!file.is_open()) return;
  const int n = O->grid.n_vox * O->desc.n_upper;
  vector<double> K((size_t) n * n);
  check(b200rt_get_influence(O->ctx, 0, B200RT_ROW_MAJOR, K.data()), O->ctx);
  write_influence(file, O->name, K, n);
}

// ---- multiplet models: O_1026_emission::define (emission/O_1026.hpp:134-217), H_lyman_multiplet::define
// (emission/H_lyman_multiplet.hpp:160-217) on the spherical grid of the facade
void observation_fit::generate_multiplet(multiplet_model &m, int kind, atmosphere_model &atm, const Real *solar,
                                         const string &atmosphere_fname, const string &sourcefn_fname) {
  if (!m.ctx) m.ctx = make_ctx();
  if (atmosphere_fname != "") atm.save(atmosphere_fname);
  atm.spherical = true;
  set_inputs &g = m.grid;
  g.plane_parallel = false;
  g.n_rb = n_radial_boundaries; g.n_sb = n_sza_boundaries; g.n_rays = n_rays_theta * n_rays_phi;
  // oxygen_RT uses rmethod_log_n_species, the Lyman multiplet models rmethod_altitude (observation_fit.cpp:41-60)
  g.rb = atm.radial_boundaries(n_radial_boundaries, kind == B200RT_MULT_O1026 ? 1 : 0);
  g.sb.assign(g.n_sb, 0); g.pts_r.assign(g.n_rb - 1, 0); g.pts_s.assign(g.n_sb - 1, 0);
  g.ray_t.assign(g.n_rays, 0); g.ray_p.assign(g.n_rays, 0); g.ray_w.assign(g.n_rays, 0);
  if (b200rt_make_grid_sph(precision, g.n_rb, g.n_sb, n_rays_theta, n_rays_phi, g.rb.data(), szamethod, 1, g.sb.data(),
                           g.pts_r.data(), g.pts_s.data(), g.ray_t.data(), g.ray_p.data(), g.ray_w.data()) != B200RT_OK)
    throw std::runtime_error("b200rt_make_grid_sph failed");
  g.n_vox = (g.n_rb - 1) * (g.n_sb - 1);
  atm.voxel_tables(g.rb, g.pts_r, g.sb, g.pts_s, g.vox);
  check(b200rt_set_grid_sph(m.ctx, g.n_rb, g.n_sb, g.n_rays, g.rb.data(), g.sb.data(), g.pts_r.data(), g.pts_s.data(),
                            g.ray_t.data(), g.ray_p.data(), g.ray_w.data()), m.ctx);
  if (b200rt_multiplet_desc_init(kind, precision, &m.desc) != B200RT_OK) throw std::runtime_error("b200rt_multiplet_desc_init failed");
  for (int l = 0; l < m.desc.n_lines; l++)
    m.desc.solar_flux[l] = (kind == B200RT_MULT_O1026 || m.desc.multiplet_index[l] == 0) ? solar[0] : solar[1];
  const int nv = g.n_vox, nl = m.desc.n_lower;
  m.T = g.vox[2]; m.T_pt = g.vox[3]; m.absb = g.vox[4]; m.absb_pt = g.vox[5];
  if (kind != B200RT_MULT_O1026) {
    if (multiplet_constant_temp) { m.T.assign(nv, multiplet_constant_temp_value); m.T_pt = m.T; }   // set_constant_temp_RT
    if (!multiplet_CO2_absorption) { m.absb.assign(nv, 0.0); m.absb_pt = m.absb; }                   // set_CO2_absorption_off
  }
  m.dens.assign((size_t) nl * nv, 0.0);
  m.dens_pt.assign((size_t) nl * nv, 0.0);
  if (kind == B200RT_MULT_O1026) {
    // Boltzmann populations of the three J levels of the ground term (O_1026.hpp:186-211; energies and weights
    // O_1026_tracker.hpp:103-110): J = 0, 1, 2 in the tracker's lower-state order
    const double erg_per_eV = 1.60218e-12;
    const double E[3] = {0.0281416 * erg_per_eV, 0.0196224 * erg_per_eV, 0.0};
    const double gw[3] = {1, 3, 5};
    for (int v = 0; v < nv; v++)
      for (int pt = 0; pt < 2; pt++) {
        const double T = pt ? m.T_pt[v] : m.T[v], bulk = pt ? g.vox[1][v] : g.vox[0][v];
        double fr[3], tot = 0;
        for (int l = 0; l < 3; l++) { fr[l] = gw[l] * std::exp(-E[l] / kB / T); tot += fr[l]; }
        for (int l = 0; l < 3; l++) (pt ? m.dens_pt : m.dens)[(size_t) l * nv + v] = fr[l] / tot * bulk;
      }
  } else {
    for (int v = 0; v < nv; v++) { m.dens[v] = g.vox[0][v]; m.dens_pt[v] = g.vox[1][v]; }
  }
  check(b200rt_set_multiplet(m.ctx, &m.desc, m.dens.data(), m.dens_pt.data(), m.T.data(), m.T_pt.data(), m.absb.data(),
                             m.absb_pt.data()), m.ctx);
  check(b200rt_generate_S(m.ctx), m.ctx);
  const int n_el = nv * m.desc.n_upper;
  m.S.assign(n_el, 0.0); m.S0.assign(n_el, 0.0);
  m.tau_sp.assign((size_t) nv * m.desc.n_lines, 0.0); m.tau_abs.assign((size_t) nv * m.desc.n_lines, 0.0);
  check(b200rt_get_solution(m.ctx, 0, m.S.data(), m.S0.data(), m.tau_sp.data(), m.tau_abs.data()), m.ctx);
  m.have_S = true;
  if (sourcefn_fname != "") {
    // grid.save_S + multiplet_CFR_emission::save (multiplet_CFR_emission.hpp:422-463)
    std::ofstream file(sourcefn_fname.c_str());
    if (file.is_open()) {
      file << "radial boundaries [cm]: " << row(g.rb) << "\n\n";
      file << "pts radii [cm]: " << row(g.pts_r) << "\n\n";
      file << "sza boundaries [rad]: " << row(g.sb) << "\n\n";
      file << "pts sza [rad]: " << row(g.pts_s) << "\n\n";
      file << "For " << m.name << "\n";
      const int ns = g.n_sb - 1, nr = g.n_rb - 1;
      auto slice = [&](const vector<double> &q, int stride, int off, int j) {
        vector<double> r(nr);
        for (int i = 0; i < nr; i++) r[i] = q[((size_t) i * ns + j) * stride + off];
        return r;
      };
      auto states = [&](const vector<double> &q, int n_states, const char *what, int j) {
        for (int st = 0; st < n_states; st++) file << "      " << what << " " << st << ": " << row(slice(q, n_states, st, j)) << "\n";
      };
      for (int j = 0; j < ns; j++) {
        file << "  For SZA = " << g.pts_s[j] << ": \n";
        file << "    Species density [cm-3]: \n";
        for (int l = 0; l < nl; l++) {
          vector<double> lev(m.dens.begin() + (size_t) l * nv, m.dens.begin() + (size_t) (l + 1) * nv);
          file << "      lower state " << l << ": " << row(slice(lev, 1, 0, j)) << "\n";
        }
        file << "    Temperature [K]: " << row(slice(m.T, 1, 0, j)) << "\n";
        file << "    Species single scattering tau: \n";
        states(m.tau_sp, m.desc.n_lines, "line", j);
        file << "    Absorber density [cm-3]: " << row(slice(m.absb, 1, 0, j)) << "\n";
        file << "    Absorber single scattering tau: \n";
        states(m.tau_abs, m.desc.n_lines, "line", j);
        file << "    Species single scattering source function S0: \n";
        states(m.S0, m.desc.n_upper, "upper state", j);
        file << "    Source function: \n";
        states(m.S, m.desc.n_upper, "upper state", j);
      }
    }
  }
}

vector<vector<observation_fit::Real>> observation_fit::multiplet_brightness(multiplet_model &m) {
  if (!m.have_S) throw std::runtime_error("observation_fit: generate a source function before asking for brightness");
  if (n_obs() == 0) throw std::runtime_error("there must be at least one observation to simulate");
  const int n = n_obs(), nl = m.desc.n_lines;
  vector<double> b((size_t) nl * n), ts((size_t) nl * n), ta((size_t) nl * n), cd((size_t) m.desc.n_lower * n);
  check(b200rt_brightness(m.ctx, n, los[0].data(), los[1].data(), los[2].data(), los[3].data(), los[4].data(), los[5].data(),
                          los[6].data(), los[7].data(), los[8].data(), 10, b.data(), ts.data(), ta.data(), cd.data()), m.ctx);
  vector<vector<Real>> r(nl);
  for (int l = 0; l < nl; l++) r[l].assign(b.begin() + (size_t) l * n, b.begin() + (size_t) (l + 1) * n);
  return r;
}

vector<observation_fit::Real> observation_fit::multiplet_source_function(int model) {
  multiplet_model *m = model == 0 ? O : model == 1 ? ly_multiplet : ly_singlet;
  if (!m || !m->have_S) throw std::runtime_error("observation_fit: no source function yet");
  return m->S;
}

void observation_fit::O_1026_generate_source_function(const Real &nOexo, const Real &Texo, const Real &solar_brightness_lyman_beta,
                                                      const string atmosphere_fname, const string sourcefn_fname) {
  const Real rmin = rMars + 100e5;       // observation_fit.cpp:669-681
  chamb_diff_1d atm(rmin, rMars + 200e5, 10.0, rmin, nOexo, CO2_exobase_density, krasnopolsky_temperature(Texo),
                    species_density_parameters::oxygen(), chamb_diff_1d::method_nspmin_nCO2exo);
  if (!O) { O = new multiplet_model; O->name = "O_1026"; }
  const Real solar[2] = {solar_brightness_lyman_beta, 0.0};
  generate_multiplet(*O, B200RT_MULT_O1026, atm, solar, atmosphere_fname, sourcefn_fname);
}
vector<vector<observation_fit::Real>> observation_fit::O_1026_brightness() {
  if (!O) throw std::runtime_error("observation_fit: generate a source function before asking for brightness");
  return multiplet_brightness(*O);
}

// The reference leaves the solar line-centre fluxes of the two Lyman multiplet models to their constructors' state
// (the set_solar_brightness call is commented out, observation_fit.cpp:752-753); the typical fluxes at Mars
// (constants.hpp:40-63) are used here.
void observation_fit::lyman_multiplet_generate_source_function(const Real &nHexo, const Real &Texo, const string atmosphere_fname,
                                                               const string sourcefn_fname) {
  chamb_diff_1d atm(nHexo, CO2_exobase_density, Texo);
  atm.copy_H_options(H_cross_section_options);
  if (!ly_multiplet) { ly_multiplet = new multiplet_model; ly_multiplet->name = "Multiplet Lyman alpha and beta"; }
  const Real solar[2] = {lyman_alpha_flux_Mars_typical, lyman_beta_flux_Mars_typical};
  generate_multiplet(*ly_multiplet, B200RT_MULT_H_LYMAN, atm, solar, atmosphere_fname, sourcefn_fname);
}
vector<vector<observation_fit::Real>> observation_fit::lyman_multiplet_brightness() {
  if (!ly_multiplet) throw std::runtime_error("observation_fit: generate a source function before asking for brightness");
  const vector<vector<Real>> lines = multiplet_brightness(*ly_multiplet);
  vector<vector<Real>> b(2, vector<Real>(n_obs()));
  for (int i = 0; i < n_obs(); i++) {
    b[0][i] = lines[0][i] + lines[1][i];     // Lyman alpha (observation_fit.cpp:786-789)
    b[1][i] = lines[2][i] + lines[3][i];     // Lyman beta
  }
  return b;
}

void observation_fit::lyman_singlet_generate_source_function(const Real &nHexo, const Real &Texo, const string atmosphere_fname,
                                                             const string sourcefn_fname) {
  chamb_diff_1d atm(nHexo, CO2_exobase_density, Texo);
  atm.copy_H_options(H_cross_section_options);
  if (!ly_singlet) { ly_singlet = new multiplet_model; ly_singlet->name = "Singlet Lyman alpha and beta"; }
  const Real solar[2] = {lyman_alpha_flux_Mars_typical, lyman_beta_flux_Mars_typical};
  generate_multiplet(*ly_singlet, B200RT_MULT_H_SINGLET, atm, solar, atmosphere_fname, sourcefn_fname);
}
vector<vector<observation_fit::Real>> observation_fit::lyman_singlet_brightness() {
  if (!ly_singlet) throw std::runtime_error("observation_fit: generate a source function before asking for brightness");
  return multiplet_brightness(*ly_singlet);
}

// ---- the sweep: every parameter set is independent (own atmosphere, own grid: rmax depends on (nH, T)),
// so sets are handed to worker threads, each owning one context (stream) on one GPU
vector<vector<vector<observation_fit::Real>>> observation_fit::brightness_batch(const vector<Real> &nHexo, const vector<Real> &Texo,
                                                                               int contexts_per_gpu, int n_gpus) {
  if (nHexo.size() != Texo.size()) throw std::invalid_argument("brightness_batch: nHexo and Texo must have the same length");
  if (n_obs() == 0) throw std::runtime_error("there must be at least one observation to simulate");
  const int n_sets = (int) nHexo.size();
  if (n_gpus <= 0) n_gpus = b200rt_device_count();
  n_gpus = std::max(1, std::min(n_gpus, b200rt_device_count()));
  const int n_workers = std::max(1, std::min(n_sets, n_gpus * std::max(1, contexts_per_gpu)));
  vector<vector<vector<Real>>> result(n_sets);
  std::atomic<int> next(0);
  vector<string> errors(n_workers);
  const auto t0 = std::chrono::steady_clock::now();
  // B200RT_BATCH_PROFILE=1: wall time per stage, summed over the worker threads (development aid)
  static const bool profile = getenv("B200RT_BATCH_PROFILE") != nullptr;
  std::atomic<long long> t_stage[5];
  for (auto &t : t_stage) t = 0;
  auto now_us = [] { return std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  auto work = [&](int w) {
    b200rt_ctx *c = nullptr;
    try {
      if (b200rt_create(w % n_gpus, precision, &c) != B200RT_OK) throw std::runtime_error("b200rt_create failed");
      bool first = true;
      set_inputs in;
      const int n = n_obs();
      vector<double> flat_B((size_t) n_hydrogen_emissions * n), flat_tab(sim_iph ? (size_t) n_hydrogen_emissions * n : 0);
      for (int i = next++; i < n_sets; i = next++) {
        long long ta = profile ? now_us() : 0;
        chamb_diff_1d atm(nHexo[i], CO2_exobase_density, Texo[i]);
        atm.copy_H_options(H_cross_section_options);
        if (profile) { const long long tb = now_us(); t_stage[0] += tb - ta; ta = tb; }
        build_inputs(atm, Texo[i], false, in);
        if (profile) { const long long tb = now_us(); t_stage[1] += tb - ta; ta = tb; }
        load_inputs(c, in);
        if (profile) { const long long tb = now_us(); t_stage[2] += tb - ta; ta = tb; }
        check(b200rt_generate_S(c), c);
        if (profile) { const long long tb = now_us(); t_stage[3] += tb - ta; ta = tb; }
        // only what the batch returns travels back: brightness, and the absorber optical depth the IPH term is extincted by
        if (first)
          check(b200rt_los_upload(c, n, los[0].data(), los[1].data(), los[2].data(), los[3].data(), los[4].data(),
                                  los[5].data(), los[6].data(), los[7].data(), los[8].data()), c);
        check(b200rt_brightness_resident(c, 10), c);
        check(b200rt_los_download(c, flat_B.data(), nullptr, sim_iph ? flat_tab.data() : nullptr, nullptr), c);
        if (profile) { const long long tb = now_us(); t_stage[4] += tb - ta; ta = tb; }
        first = false;
        vector<vector<Real>> &out = result[i];
        out.assign(n_hydrogen_emissions, vector<Real>());
        for (int e = 0; e < n_hydrogen_emissions; e++) {
          out[e].assign(flat_B.begin() + (size_t) e * n, flat_B.begin() + (size_t) (e + 1) * n);
          if (sim_iph)
            for (int k = 0; k < n; k++) {
              const Real ta = flat_tab[(size_t) e * n + k];
              out[e][k] += (ta != -1) ? iph_unextincted[k][e] * std::exp(-ta) : 0.0;
            }
        }
      }
    } catch (const std::exception &ex) {
      errors[w] = ex.what();
    }
    b200rt_destroy(c);
  };
  vector<std::thread> pool;
  for (int w = 0; w < n_workers; w++) pool.emplace_back(work, w);
  for (auto &t : pool) t.join();
  batch_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  if (profile)
    fprintf(stderr, "brightness_batch: %d sets, %d workers, %.3f s wall; per set (ms, thread time): atmosphere %.3f  build_inputs %.3f  "
            "load_inputs %.3f  generate_S %.3f  brightness %.3f\n", n_sets, n_workers, batch_seconds,
            t_stage[0] / 1e3 / n_sets, t_stage[1] / 1e3 / n_sets, t_stage[2] / 1e3 / n_sets, t_stage[3] / 1e3 / n_sets,
            t_stage[4] / 1e3 / n_sets);
  for (auto &e : errors)
    if (!e.empty()) throw std::runtime_error("brightness_batch: " + e);
  return result;
}
