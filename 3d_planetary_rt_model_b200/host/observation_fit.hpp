// observation_fit.hpp -- host facade with the public interface of the reference's observation_fit
// (src/observation_fit.hpp:23-389), implemented on the C ABI of include/b200rt.h.  Plain C++ (g++); nothing here needs
// nvcc.  Every member the reference's Cython binding declares (python/py_corona_sim.pyx:33-172) exists here with the
// same name and argument list, so that binding compiles UNCHANGED against this header (oracle/Makefile `pyx`,
// tests/test_pyx_dropin.py).
//
// What each member maps to (reference src/):
//   add_observation            observation_fit.cpp:62-66 + observation::add_MSO_observation (observation.hpp:46-65)
//   set_g_factor               observation_fit.cpp:74-92
//   simulate_iph, add_observation_ra_dec, get_unextincted_iph        observation_fit.cpp:94-119
//   generate_source_function   observation_fit.cpp:122-169 -> generate_source_function_sph_azi_sym (hpp:241-294)
//                              / generate_source_function_plane_parallel (hpp:189-239)
//   ..._lc, ..._effv           observation_fit.cpp:171-197 (Temp_converter, chamberlain_exosphere.hpp:45-75)
//   ..._variable_thermosphere  observation_fit.cpp:200-262
//   ..._nH_asym, ..._temp_asym observation_fit.cpp:264-358
//   ..._tabular_atmosphere     observation_fit.cpp:360-411
//   set_use_CO2_absorption ... observation_fit.cpp:413-487
//   brightness & friends       observation_fit.cpp:491-637 (H), 591-637 (D)
//   save_influence_matrix[_O_1026]            observation_fit.cpp:647-653
//   O_1026_*, lyman_multiplet_*, lyman_singlet_*          observation_fit.cpp:656-868
// Like the reference, every model (H, D, their plane-parallel twins, O I 102.6, the two Lyman multiplet models) keeps
// its own RT state: here one b200rt context each, created on first use.
// New (SURVEY.md 8(f) N1): brightness_batch() runs a whole (nH, T) sweep -- one atmosphere, grid, source function and
// brightness per parameter set -- over all GPUs with several contexts each, instead of the reference's Python loop over
// generate_source_function + brightness.
#pragma once
#include <fstream>
#include <string>
#include <vector>
#include "atmosphere.hpp"

struct b200rt_ctx;

class observation_fit {
public:
  typedef b200rt_host::Real Real;
  static const int n_radial_boundaries = 40;   // observation_fit.hpp:44-47 (standard resolution case)
  static const int n_sza_boundaries = 20;
  static const int n_rays_theta = 7;
  static const int n_rays_phi = 12;
  static const int n_rays_pp = 7;              // plane_parallel_grid<n_radial_boundaries, 7>, observation_fit.hpp:48-50
  static const int n_hydrogen_emissions = 2;
  static const int n_voxels = (n_radial_boundaries - 1) * (n_sza_boundaries - 1);

  explicit observation_fit(const std::string iph_sfn_fnamee, int device = -1,   // -1: every visible GPU (one handle)
                           bool single_precision = false);                     // device arithmetic in float (the reference GPU build's Real)
  ~observation_fit();
  observation_fit(const observation_fit &) = delete;
  observation_fit &operator=(const observation_fit &) = delete;

  b200rt_host::Temp_converter Tconv;           // also the source of the H escape fraction

  void add_observation(const std::vector<std::vector<Real>> &MSO_locations,
                       const std::vector<std::vector<Real>> &MSO_directions);
  // the same from flat [n][3] arrays: what a buffer-protocol caller (the Cython fast path, host/py_corona_sim_b200.pyx)
  // hands over without building 2 n small vectors
  void add_observation(const double *MSO_locations, const double *MSO_directions, int n);
  void get_unextincted_iph();
  void set_g_factor(std::vector<Real> &g);
  void simulate_iph(const bool sim_iphh);
  void add_observation_ra_dec(const std::vector<Real> &mars_ecliptic_coords, const std::vector<Real> &RAA,
                              const std::vector<Real> &Decc);

  void generate_source_function(const Real &nHexo, const Real &Texo, const std::string atmosphere_fname = "",
                                const std::string sourcefn_fname = "", const bool plane_parallel = false,
                                const bool deuterium = false);
  void generate_source_function_effv(const Real &nHexo, const Real &effv_exo, const std::string atmosphere_fname = "",
                                     const std::string sourcefn_fname = "", const bool plane_parallel = false,
                                     const bool deuterium = false);
  void generate_source_function_lc(const Real &nHexo, const Real &lc_exo, const std::string atmosphere_fname = "",
                                   const std::string sourcefn_fname = "", const bool plane_parallel = false,
                                   const bool deuterium = false);
  void generate_source_function_variable_thermosphere(const Real &nHexo, const Real &Texo, const Real &nCO2rminn,
                                                      const Real rexoo, const Real rminn, const Real rmaxx,
                                                      const Real rmindiffusionn, const Real T_tropo, const Real r_tropo,
                                                      const Real shape_parameter, const std::string atmosphere_fname = "",
                                                      const std::string sourcefn_fname = "",
                                                      const bool plane_parallel = false, const bool deuterium = false);
  void generate_source_function_nH_asym(const Real &nHexo, const Real &Texo, const Real &asym,
                                        const std::string sourcefn_fname = "", const bool deuterium = false);
  void generate_source_function_temp_asym(const Real &nHavg, const Real &Tnoon, const Real &Tmidnight,
                                          const std::string sourcefn_fname = "", const bool deuterium = false);
  void generate_source_function_temp_asym(const Real &nHavg, const Real &Tnoon, const Real &Tmidnight,
                                          const Real nCO2rminn, const Real rexoo, const Real rminn, const Real rmaxx,
                                          const Real rmindiffusionn, const Real T_tropo, const Real r_tropo,
                                          const Real shape_parameter, const Real Tpowerr,
                                          const std::string sourcefn_fname = "", const bool deuterium = false);
  void generate_source_function_tabular_atmosphere(const Real rmin, const Real rexo, const Real rmax,
                                                   const std::vector<double> &alt_nH, const std::vector<double> &log_nH,
                                                   const std::vector<double> &alt_nCO2, const std::vector<double> &log_nCO2,
                                                   const std::vector<double> &alt_temp, const std::vector<double> &temp,
                                                   const bool compute_exosphere = false, const bool plane_parallel = false,
                                                   const bool deuterium = false, const std::string sourcefn_fname = "");

  void set_use_CO2_absorption(const bool use_CO2_absorption = true);
  void set_use_temp_dependent_sH(const bool use_temp_dependent_sH = true, const Real constant_temp_sH = -1);
  void set_sza_method_uniform();
  void set_sza_method_uniform_cos();
  void reset_H_lya_xsec_coef(const Real xsec_coef = b200rt_host::lyman_alpha_line_center_cross_section_coef);
  void reset_H_lyb_xsec_coef(const Real xsec_coef = b200rt_host::lyman_beta_line_center_cross_section_coef);
  void reset_CO2_lya_xsec(const Real xsec = b200rt_host::CO2_lyman_alpha_absorption_cross_section);
  void reset_CO2_lyb_xsec(const Real xsec = b200rt_host::CO2_lyman_beta_absorption_cross_section);
  Real get_CO2_exobase_density();
  void reset_CO2_exobase_density();
  void set_CO2_exobase_density(const double nCO2);

  void save_influence_matrix(const std::string fname);
  void save_influence_matrix_O_1026(const std::string fname);

  void set_H_density_tweak(const bool tweak_H_densityy);
  void set_H_density_tweak_values(const std::vector<int> voxels_to_tweak, const Real tweak_factor);
  void set_H_temp_tweak(const bool tweak_H_tempp);
  void set_H_temp_tweak_values(const std::vector<int> voxels_to_tweak, const Real tweak_factor);

  std::vector<std::vector<Real>> brightness();
  std::vector<std::vector<Real>> species_col_dens();
  std::vector<std::vector<Real>> tau_species_final();
  std::vector<std::vector<Real>> tau_absorber_final();
  std::vector<std::vector<Real>> iph_brightness_observed();
  std::vector<std::vector<Real>> iph_brightness_unextincted();

  std::vector<std::vector<Real>> D_brightness();
  std::vector<std::vector<Real>> D_col_dens();
  std::vector<std::vector<Real>> tau_D_final();

  void O_1026_generate_source_function(const Real &nOexo, const Real &Texo, const Real &solar_brightness_lyman_beta,
                                       const std::string atmosphere_fname = "", const std::string sourcefn_fname = "");
  std::vector<std::vector<Real>> O_1026_brightness();
  void lyman_multiplet_generate_source_function(const Real &nHexo, const Real &Texo,
                                                const std::string atmosphere_fname = "",
                                                const std::string sourcefn_fname = "");
  std::vector<std::vector<Real>> lyman_multiplet_brightness();
  void lyman_singlet_generate_source_function(const Real &nHexo, const Real &Texo, const std::string atmosphere_fname = "",
                                              const std::string sourcefn_fname = "");
  std::vector<std::vector<Real>> lyman_singlet_brightness();

  // ---- batched sweep: result[i_set][i_emission][i_obs] = brightness (incl. extincted IPH if simulated)
  std::vector<std::vector<std::vector<Real>>> brightness_batch(const std::vector<Real> &nHexo, const std::vector<Real> &Texo,
                                                               int contexts_per_gpu = 4, int n_gpus = -1);
  double last_batch_seconds() const { return batch_seconds; }

  // ---- access to the solution of the last generate_source_function* of the H (which = 0), D (1), plane-parallel H (2)
  // and plane-parallel D (3) models: what save_S writes
  std::vector<Real> source_function(int i_emission, int which = 0);
  std::vector<Real> radial_boundaries(int which = 0) const;
  // source function of the multiplet models (0 = O I 102.6, 1 = Lyman multiplet, 2 = Lyman singlet): [n_vox * n_upper]
  std::vector<Real> multiplet_source_function(int model);
  int n_obs() const { return (int) los[0].size(); }

  // ---- line-of-sight weighting functions of the H (which = 0) or D (1) model for the current observations, with
  // n_subsamples = 10 like brightness(): W (n_obs x n_vox, CSR) with W * source_function(e, which) = brightness()[e]
  // without the IPH term.  The plane-parallel models (2, 3) have no brightness and throw.
  struct csr_matrix {
    int n_rows = 0, n_cols = 0;
    std::vector<long long> indptr;   // [n_rows + 1]
    std::vector<int> indices;        // [nnz] voxel ids, ascending within a row
    std::vector<Real> data;          // [nnz]
  };
  csr_matrix brightness_weights(int i_emission, int which = 0);
  // d(sum_l obs_weights[l] * brightness()[i_emission][l]) / dS0 over the voxels of the H (0) or D (1) model: W^T w,
  // then one adjoint solve on the model's influence matrix, (I - w K)^T lambda = W^T w, so that the weighted brightness
  // changes by lambda . dS0 for a change dS0 of the single-scattering source.  The IPH term does not depend on S0.
  // obs_weights has one entry per observation; the plane-parallel models (2, 3) throw.
  std::vector<Real> brightness_source_sensitivity(int i_emission, const std::vector<Real> &obs_weights, int which = 0);

private:
  struct set_inputs;       // grid + the eight tables of each emission for one parameter set
  struct singlet_model;    // one RT_grid<singlet_CFR, 2, grid> of the reference + its observation outputs
  struct multiplet_model;  // one RT_grid<multiplet emission, 1, grid>
  void build_inputs(const b200rt_host::atmosphere_model &atm, const Real &Texo, bool plane_parallel, set_inputs &in) const;
  void load_inputs(b200rt_ctx *c, const set_inputs &in) const;
  void run_brightness(b200rt_ctx *c, bool upload, std::vector<std::vector<Real>> (&q)[4]) const;
  void generate(b200rt_host::atmosphere_model &atm, const Real &Texo, bool plane_parallel, bool deuterium,
                const std::string &atmosphere_fname, const std::string &sourcefn_fname);
  void model_brightness(singlet_model &m);
  void generate_multiplet(multiplet_model &m, int kind, b200rt_host::atmosphere_model &atm, const Real *solar,
                          const std::string &atmosphere_fname, const std::string &sourcefn_fname);
  std::vector<std::vector<Real>> multiplet_brightness(multiplet_model &m);
  b200rt_ctx *make_ctx() const;
  void check(int rc, b200rt_ctx *c) const;
  void save_S(const std::string &fname, const set_inputs &in);

  int device;
  int precision;           // B200RT_F64 or B200RT_F32: arithmetic of the device kernels
  b200rt_host::H_cross_sections H_cross_section_options;
  const Real default_CO2_exobase_density = 2e8;
  Real CO2_exobase_density;
  int szamethod = 1;                   // szamethod_uniform_cos (observation_fit.cpp:37)
  Real g_factor[n_hydrogen_emissions];
  std::string iph_sfn_fname;
  bool sim_iph = false, iph_table_loaded = false;
  bool tweak_H_density = false, tweak_H_temp = false;
  std::vector<int> tweak_H_density_voxel_numbers, tweak_H_temp_voxel_numbers;
  Real tweak_H_density_factor = 1.0, tweak_H_temp_factor = 1.0;
  bool multiplet_CO2_absorption = true, multiplet_constant_temp = false;
  Real multiplet_constant_temp_value = -1;

  // observation (observation.hpp): geometry as the nine atmo_vector fields, shared by every model
  std::vector<Real> los[9];
  std::vector<Real> mars_ecliptic_pos, ra, dec;
  std::vector<std::vector<Real>> iph_unextincted;   // [i_obs][i_emission]
  singlet_model *H = nullptr, *D = nullptr, *H_pp = nullptr, *D_pp = nullptr;
  multiplet_model *O = nullptr, *ly_multiplet = nullptr, *ly_singlet = nullptr;
  singlet_model &singlet(int which);
  double batch_seconds = 0;
};
// the ASCII writers on plain arrays (what save_S / save_influence_matrix print; observation_fit.cpp), exposed so that
// their output can be compared byte for byte with the reference's own writers
void write_S_file(const std::string &fname, bool plane_parallel, int n_rb, int n_sb, const std::vector<double> &rb,
                  const std::vector<double> &pts_r, const std::vector<double> &sb, const std::vector<double> &pts_s, int n_em,
                  const std::vector<std::string> &names, const std::vector<std::vector<std::vector<double>>> &q);
void write_influence(std::ofstream &file, const std::string &name, const std::vector<double> &K, int n);


