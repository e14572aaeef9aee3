// b200rt_api.cu -- the C ABI (include/b200rt.h): context lifetime, argument checks, device-group dispatch.  The work behind
// each entry point lives in api_source_function.cu / api_brightness.cu / api_traverse.cu / api_multiplet.cu / iph.cu /
// device_group.cu (see api_internal.hpp).  Host code only.
#include "api_internal.hpp"

using namespace b200rt;
using namespace b200rt::api;

// a context made by b200rt_create_multi owns no device state itself: every call fans out to its members (device_group.cu)
#define GROUP_DISPATCH(c, call) do { if ((c)->group) return call; } while (0)

// ====================================================================== C ABI
extern "C" {

int b200rt_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int b200rt_create(int device, int precision, b200rt_ctx **out) {
  if (!out || (precision != B200RT_F64 && precision != B200RT_F32)) return B200RT_ERR_ARG;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return B200RT_ERR_CUDA;  // no CPU fallback
  if (cudaSetDevice(device) != cudaSuccess) return B200RT_ERR_CUDA;
  b200rt_ctx *c = new (std::nothrow) b200rt_ctx;
  if (!c) return B200RT_ERR_NOMEM;
  c->device = device;
  c->precision = precision;
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return B200RT_ERR_CUDA; }
  if (c->work_counter.ensure(4 * sizeof(int)) != cudaSuccess || c->step_counter.ensure(sizeof(unsigned long long)) != cudaSuccess) {
    delete c;
    return B200RT_ERR_CUDA;
  }
  *out = c;
  return B200RT_OK;
}

int b200rt_destroy(b200rt_ctx *c) {
  if (!c) return B200RT_OK;
  if (c->group) return group_destroy(c);
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  DevBuf *bufs[] = {&c->grid_tables, &c->sun_rays, &c->list_dist, &c->list_ent, &c->list_len, &c->list_flag,
                    &c->work_counter, &c->step_counter, &c->los_in, &c->los_out, &c->los_order, &c->lu, &c->lu_dinv, &c->lu_flag,
                    &c->iph.dev, &c->iph.io, &c->vox_map, &c->sph_table, &c->kry_xchg, &c->kry_work, &c->kry_bp,
                    &c->kry_adj_xchg, &c->kry_adj_work, &c->kry_kt, &c->kry_adj_io,
                    &c->lw.row_ptr, &c->lw.row_cnt, &c->lw.col, &c->lw.val, &c->lw.rec, &c->lw.scratch, &c->lw.xy};
  for (DevBuf *b : bufs) b->release();
  c->host_scratch.release();
  c->host_words.release();
  c->host_out.release();
  c->host_stage.release();
  c->dev_stage.release();
  for (int e = 0; e < MAX_EMISSIONS; e++) {
    Emission &E = c->em[e];
    DevBuf *eb[] = {&E.tabs, &E.phi, &E.mrec, &E.K, &E.S0, &E.tau_sp, &E.tau_abs, &E.S, &E.S_real, &E.rec_pt, &E.rec_avg};
    for (DevBuf *b : eb) b->release();
  }
  {
    Multiplet &M = c->mult;
    DevBuf *mb[] = {&M.tabs, &M.rec_step, &M.rec_org, &M.rec_w0, &M.tsv, &M.tav, &M.K, &M.S0, &M.tau_sp, &M.tau_abs, &M.S,
                    &M.S_real, &M.rec_pt, &M.rec_avg};
    for (DevBuf *b : mb) b->release();
  }
  if (c->grid_view) ::operator delete(c->grid_view);
  if (c->march_view) ::operator delete(c->march_view);
  for (cudaEvent_t ev : c->lu_events) cudaEventDestroy(ev);
  for (cudaEvent_t ev : c->timer_events) cudaEventDestroy(ev);
  if (c->lu_graph) cudaGraphExecDestroy(c->lu_graph);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->out_stream) cudaStreamDestroy(c->out_stream);
  if (c->ev_rows) cudaEventDestroy(c->ev_rows);
  if (c->stream2) cudaStreamDestroy(c->stream2);
  if (c->stream3) cudaStreamDestroy(c->stream3);
  cudaStreamDestroy(c->stream);
  delete c;
  return B200RT_OK;
}

const char *b200rt_last_error(const b200rt_ctx *c) { return c ? c->err.c_str() : "null context"; }

int b200rt_synchronize(b200rt_ctx *c) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_synchronize(c));
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  return B200RT_OK;
}

int b200rt_make_grid_sph(int precision, int n_rb, int n_sb, int n_theta, int n_phi, const double *rb, int szamethod,
                         int raymethod, double *sb, double *pts_r, double *pts_s, double *ray_t, double *ray_p,
                         double *ray_domega) {
  if (n_rb < 2 || n_sb < 3 || n_theta < 2 || n_phi < 1 || !rb) return B200RT_ERR_ARG;
  if (precision == B200RT_F64) make_grid_sph<double>(n_rb, n_sb, n_theta, n_phi, rb, szamethod, raymethod, sb, pts_r, pts_s, ray_t, ray_p, ray_domega);
  else make_grid_sph<float>(n_rb, n_sb, n_theta, n_phi, rb, szamethod, raymethod, sb, pts_r, pts_s, ray_t, ray_p, ray_domega);
  return B200RT_OK;
}

int b200rt_fold_rays(int precision, int n_rays, const double *ray_t, const double *ray_p, const double *ray_domega,
                     int *rep, int *n_marched) {
  if (n_rays < 1 || !ray_t || !ray_p || !ray_domega || !rep || !n_marched) return B200RT_ERR_ARG;
  *n_marched = precision == B200RT_F64 ? fold_rays<double>(n_rays, ray_t, ray_p, ray_domega, rep)
                                       : fold_rays<float>(n_rays, ray_t, ray_p, ray_domega, rep);
  return B200RT_OK;
}

int b200rt_set_grid_sph(b200rt_ctx *c, int n_rb, int n_sb, int n_rays, const double *rb, const double *sb,
                        const double *pts_r, const double *pts_s, const double *ray_t, const double *ray_p,
                        const double *ray_domega) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_set_grid_sph(c, n_rb, n_sb, n_rays, rb, sb, pts_r, pts_s, ray_t, ray_p, ray_domega));
  if (n_rb < 2 || n_sb < 3 || n_rays < 1 || !rb || !sb || !pts_r || !pts_s || !ray_t || !ray_p || !ray_domega)
    return fail(c, B200RT_ERR_ARG, "b200rt_set_grid_sph: bad argument");
  cudaSetDevice(c->device);
  HostGrid &h = c->hg;
  h.pp = false;
  h.n_rb = n_rb; h.n_sb = n_sb; h.n_vox = (n_rb - 1) * (n_sb - 1); h.n_rays = n_rays; h.cap = 2 * n_rb + n_sb;
  h.rb.assign(rb, rb + n_rb); h.sb.assign(sb, sb + n_sb);
  h.pts_r.assign(pts_r, pts_r + n_rb - 1); h.pts_s.assign(pts_s, pts_s + n_sb - 1);
  h.ray_t.assign(ray_t, ray_t + n_rays); h.ray_p.assign(ray_p, ray_p + n_rays);
  h.ray_domega.assign(ray_domega, ray_domega + n_rays);
  int rc = is64(c) ? upload_grid<double>(c) : upload_grid<float>(c);
  if (rc) return rc;
  c->have_grid = true;
  c->n_em = 0;
  for (int e = 0; e < 2; e++) { c->row_sink[e] = nullptr; c->row_sink_n_vox[e] = 0; }   // named for the old geometry
  for (int e = 0; e < MAX_EMISSIONS; e++) { c->em[e].defined = c->em[e].have_K = c->em[e].have_S = false; }
  c->mult.defined = c->mult.have_K = c->mult.have_S = false;
  c->lw.valid = false;
  return B200RT_OK;
}

int b200rt_make_grid_pp(int precision, int n_rb, int n_theta, const double *rb, double *pts_r, double *ray_t,
                        double *ray_domega) {
  if (n_rb < 2 || n_theta < 1 || !rb || !pts_r || !ray_t || !ray_domega) return B200RT_ERR_ARG;
  if (precision == B200RT_F64) make_grid_pp<double>(n_rb, n_theta, rb, pts_r, ray_t, ray_domega);
  else make_grid_pp<float>(n_rb, n_theta, rb, pts_r, ray_t, ray_domega);
  return B200RT_OK;
}

int b200rt_set_grid_pp(b200rt_ctx *c, int n_rb, int n_rays, const double *rb, const double *pts_r,
                       const double *ray_t, const double *ray_domega) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_set_grid_pp(c, n_rb, n_rays, rb, pts_r, ray_t, ray_domega));
  if (n_rb < 2 || n_rays < 1 || !rb || !pts_r || !ray_t || !ray_domega)
    return fail(c, B200RT_ERR_ARG, "b200rt_set_grid_pp: bad argument");
  cudaSetDevice(c->device);
  HostGrid &h = c->hg;
  // one SZA column [0, pi] whose voxel points sit on the +z axis (pt.xyz(0,0,pts_radii[i]) => pt.t = 0,
  // grid_plane_parallel.hpp:189-204); rays have phi = 0 (:219)
  h.pp = true;
  h.n_rb = n_rb; h.n_sb = 2; h.n_vox = n_rb - 1; h.n_rays = n_rays; h.cap = 2 * n_rb + 2;
  h.rb.assign(rb, rb + n_rb); h.sb.assign({0.0, M_PI});
  h.pts_r.assign(pts_r, pts_r + n_rb - 1); h.pts_s.assign(1, 0.0);
  h.ray_t.assign(ray_t, ray_t + n_rays); h.ray_p.assign(n_rays, 0.0);
  h.ray_domega.assign(ray_domega, ray_domega + n_rays);
  int rc = is64(c) ? upload_grid<double>(c) : upload_grid<float>(c);
  if (rc) return rc;
  c->have_grid = true;
  c->n_em = 0;
  for (int e = 0; e < 2; e++) { c->row_sink[e] = nullptr; c->row_sink_n_vox[e] = 0; }   // named for the old geometry
  for (int e = 0; e < MAX_EMISSIONS; e++) { c->em[e].defined = c->em[e].have_K = c->em[e].have_S = false; }
  c->mult.defined = c->mult.have_K = c->mult.have_S = false;
  c->lw.valid = false;
  return B200RT_OK;
}

int b200rt_set_singlet(b200rt_ctx *c, int e, int n_em, double branching, double T_ref, double sigma_ref, double g,
                       const double *T_ratio, const double *density, const double *dtau_species,
                       const double *dtau_absorber, const double *T_ratio_pt, const double *density_pt,
                       const double *dtau_species_pt, const double *dtau_absorber_pt) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_set_singlet(c, e, n_em, branching, T_ref, sigma_ref, g, T_ratio, density, dtau_species, dtau_absorber, T_ratio_pt, density_pt, dtau_species_pt, dtau_absorber_pt));
  if (!c->have_grid) return fail(c, B200RT_ERR_STATE, "set the grid before the emissions");
  if (n_em < 1 || n_em > MAX_EMISSIONS || e < 0 || e >= n_em) return fail(c, B200RT_ERR_ARG, "bad emission index");
  const double *arr[8] = {T_ratio, density, dtau_species, dtau_absorber, T_ratio_pt, density_pt, dtau_species_pt, dtau_absorber_pt};
  for (auto p : arr) if (!p) return fail(c, B200RT_ERR_ARG, "null emission table");
  cudaSetDevice(c->device);
  c->n_em = n_em;
  c->mult.defined = false;
  c->lw.valid = false;
  Emission &E = c->em[e];
  E.branching = branching; E.T_ref = T_ref; E.sigma_ref = sigma_ref; E.g_factor = g;
  int rc = api::set_singlet(c, e, arr);
  if (rc) return rc;
  E.defined = true; E.have_K = false; E.have_S = false; E.residual = -1;
  return B200RT_OK;
}

int b200rt_multiplet_desc_init(int kind, int precision, b200rt_multiplet_desc *d) {
  if (!d || (precision != B200RT_F64 && precision != B200RT_F32)) return B200RT_ERR_ARG;
  return precision == B200RT_F64 ? multiplet_desc_init<double>(kind, d) : multiplet_desc_init<float>(kind, d);
}

int b200rt_set_multiplet(b200rt_ctx *c, const b200rt_multiplet_desc *d, const double *species_density,
                         const double *species_density_pt, const double *species_T, const double *species_T_pt,
                         const double *absorber_density, const double *absorber_density_pt) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_set_multiplet(c, d, species_density, species_density_pt, species_T, species_T_pt, absorber_density, absorber_density_pt));
  if (!c->have_grid) return fail(c, B200RT_ERR_STATE, "set the grid before the emissions");
  const double *arr[6] = {species_density, species_density_pt, species_T, species_T_pt, absorber_density, absorber_density_pt};
  for (auto p : arr) if (!p) return fail(c, B200RT_ERR_ARG, "null emission table");
  if (!d || mult_check_desc(*d))
    return fail(c, B200RT_ERR_ARG, "multiplet descriptor does not match the line / level tables of its kind");
  cudaSetDevice(c->device);
  c->n_em = 0;
  c->lw.valid = false;
  for (int e = 0; e < 2; e++) { c->row_sink[e] = nullptr; c->row_sink_n_vox[e] = 0; }
  for (int e = 0; e < MAX_EMISSIONS; e++) { c->em[e].defined = c->em[e].have_K = c->em[e].have_S = false; }
  Multiplet &M = c->mult;
  M.d = *d;
  M.defined = false;
  int rc = api::set_multiplet(c, arr);
  if (rc) return rc;
  M.defined = true; M.have_K = false; M.have_S = false; M.residual = -1; M.rec_dirty = true;
  return B200RT_OK;
}

int b200rt_set_g_factor(b200rt_ctx *c, int e, double g) {
  if (!c || e < 0 || e >= MAX_EMISSIONS) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_set_g_factor(c, e, g));
  c->em[e].g_factor = g;
  c->lw.valid = false;
  return B200RT_OK;
}

int b200rt_influence(b200rt_ctx *c, int v_begin, int v_end) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_influence(c, 1, &v_begin, &v_end));
  if (!c->have_grid || (c->n_em < 1 && !c->mult.defined)) return fail(c, B200RT_ERR_STATE, "grid / emissions not set");
  if (v_begin < 0 || v_end > c->hg.n_vox || v_begin > v_end) return fail(c, B200RT_ERR_ARG, "bad voxel range");
  cudaSetDevice(c->device);
  const std::vector<std::pair<int, int>> one = {{v_begin, v_end}};
  if (c->mult.defined) return api::mult_influence(c, one);
  return api::influence(c, one);
}

int b200rt_influence_ranges(b200rt_ctx *c, int n_ranges, const int *v_begin, const int *v_end) {
  if (!c || n_ranges < 0 || (n_ranges > 0 && (!v_begin || !v_end))) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_influence(c, n_ranges, v_begin, v_end));
  if (!c->have_grid || (c->n_em < 1 && !c->mult.defined)) return fail(c, B200RT_ERR_STATE, "grid / emissions not set");
  std::vector<std::pair<int, int>> r;
  int last_end = 0;
  for (int i = 0; i < n_ranges; i++) {
    if (v_begin[i] < last_end || v_end[i] > c->hg.n_vox || v_begin[i] > v_end[i])
      return fail(c, B200RT_ERR_ARG, "voxel ranges must be ascending, disjoint and inside the grid");
    last_end = v_end[i];
    r.emplace_back(v_begin[i], v_end[i]);
  }
  cudaSetDevice(c->device);
  if (c->mult.defined) return api::mult_influence(c, r);
  return api::influence(c, r);
}

int b200rt_solve(b200rt_ctx *c) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_solve(c));
  cudaSetDevice(c->device);
  if (c->mult.defined) return api::mult_solve(c, true);
  return api::solve(c, true);
}

int b200rt_generate_S(b200rt_ctx *c) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_generate_S(c));
  int rc = b200rt_influence(c, 0, c->hg.n_vox);
  if (rc) return rc;
  if (c->mult.defined) return api::mult_solve(c, false);
  return api::solve(c, false);
}

int b200rt_last_step_count(b200rt_ctx *c, long long *n) {
  if (!c || !n) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_counts(c, 0, n));
  *n = c->last_steps;
  return B200RT_OK;
}

int b200rt_last_substep_count(b200rt_ctx *c, long long *n) {
  if (!c || !n) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_counts(c, 1, n));
  *n = c->last_substeps;
  return B200RT_OK;
}

int b200rt_get_solution(b200rt_ctx *c, int e, double *S, double *S0, double *tsp, double *tab) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_forward(c, b200rt_get_solution(group_owner(c, e), e, S, S0, tsp, tab)));
  if (c->mult.defined) {
    if (e != 0) return B200RT_ERR_ARG;
    cudaSetDevice(c->device);
    Multiplet &M = c->mult;
    const size_t ne = (size_t) c->hg.n_vox * M.d.n_upper * sizeof(double), nl = (size_t) c->hg.n_vox * M.d.n_lines * sizeof(double);
    if (S) {
      if (!M.have_S) return fail(c, B200RT_ERR_STATE, "source function not solved");
      B200RT_CUDA(c, cudaMemcpyAsync(S, M.S.p, ne, cudaMemcpyDeviceToHost, c->stream));
    }
    if ((S0 || tsp || tab) && !M.have_K) return fail(c, B200RT_ERR_STATE, "influence pass not run");
    if (S0) B200RT_CUDA(c, cudaMemcpyAsync(S0, M.S0.p, ne, cudaMemcpyDeviceToHost, c->stream));
    if (tsp) B200RT_CUDA(c, cudaMemcpyAsync(tsp, M.tau_sp.p, nl, cudaMemcpyDeviceToHost, c->stream));
    if (tab) B200RT_CUDA(c, cudaMemcpyAsync(tab, M.tau_abs.p, nl, cudaMemcpyDeviceToHost, c->stream));
    B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
    return B200RT_OK;
  }
  if (e < 0 || e >= c->n_em) return B200RT_ERR_ARG;
  cudaSetDevice(c->device);
  Emission &E = c->em[e];
  const size_t n = (size_t) c->hg.n_vox, nb = n * sizeof(double);
  if (S && !E.have_S) return fail(c, B200RT_ERR_STATE, "source function not solved");
  if ((S0 || tsp || tab) && !E.have_K) return fail(c, B200RT_ERR_STATE, "influence pass not run");
  // through page-locked staging: a copy into the caller's (pageable) arrays would block inside the runtime under a lock
  // that stalls the other contexts of the process (common.hpp, PinnedBuf)
  B200RT_CUDA(c, c->host_stage.ensure(4 * nb));
  double *hs = c->host_stage.as<double>();
  double *dst[4] = {S, S0, tsp, tab};
  const void *src[4] = {E.S.p, E.S0.p, E.tau_sp.p, E.tau_abs.p};
  for (int q = 0; q < 4; q++)
    if (dst[q]) B200RT_CUDA(c, cudaMemcpyAsync(hs + q * n, src[q], nb, cudaMemcpyDeviceToHost, c->stream));
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  for (int q = 0; q < 4; q++)
    if (dst[q]) std::memcpy(dst[q], hs + q * n, nb);
  return B200RT_OK;
}

int b200rt_get_influence(b200rt_ctx *c, int e, int layout, double *K) {
  if (!c || !K) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_forward(c, b200rt_get_influence(group_owner_K(c, e), e, layout, K)));
  const bool mm = c->mult.defined;
  if (mm ? e != 0 : (e < 0 || e >= c->n_em)) return B200RT_ERR_ARG;
  cudaSetDevice(c->device);
  if (!(mm ? c->mult.have_K : c->em[e].have_K)) return fail(c, B200RT_ERR_STATE, "influence matrix not built");
  const size_t n = mm ? (size_t) c->hg.n_vox * c->mult.d.n_upper : (size_t) c->hg.n_vox;
  const void *Kdev = mm ? c->mult.K.p : c->em[e].K.p;
  if (layout == B200RT_ROW_MAJOR) {
    B200RT_CUDA(c, cudaMemcpyAsync(K, Kdev, n * n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  } else {
    std::vector<double> tmp(n * n);
    B200RT_CUDA(c, cudaMemcpyAsync(tmp.data(), Kdev, n * n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
    for (size_t i = 0; i < n; i++) for (size_t j = 0; j < n; j++) K[j * n + i] = tmp[i * n + j];
  }
  return B200RT_OK;
}

int b200rt_set_sourcefn(b200rt_ctx *c, int e, const double *S) {
  if (!c || !S) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_set_sourcefn(c, e, S));
  if (c->mult.defined) {
    if (e != 0) return B200RT_ERR_ARG;
    cudaSetDevice(c->device);
    Multiplet &M = c->mult;
    const int ne = c->hg.n_vox * M.d.n_upper;
    B200RT_CUDA(c, cudaMemcpyAsync(M.S.p, S, ne * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    if (is64(c)) B200RT_CUDA(c, launch_convert<double>(M.S.as<double>(), M.S_real.as<double>(), ne, c->stream));
    else B200RT_CUDA(c, launch_convert<float>(M.S.as<double>(), M.S_real.as<float>(), ne, c->stream));
    B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
    M.have_S = true;
    M.rec_dirty = true;
    return B200RT_OK;
  }
  if (e < 0 || e >= c->n_em) return B200RT_ERR_ARG;
  cudaSetDevice(c->device);
  Emission &E = c->em[e];
  if (!E.defined) return fail(c, B200RT_ERR_STATE, "emission not defined");
  const int n = c->hg.n_vox;
  B200RT_CUDA(c, c->host_stage.ensure((size_t) n * sizeof(double)));
  std::memcpy(c->host_stage.p, S, (size_t) n * sizeof(double));
  B200RT_CUDA(c, cudaMemcpyAsync(E.S.p, c->host_stage.p, n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  if (is64(c)) B200RT_CUDA(c, launch_convert<double>(E.S.as<double>(), E.S_real.as<double>(), n, c->stream));
  else B200RT_CUDA(c, launch_convert<float>(E.S.as<double>(), E.S_real.as<float>(), n, c->stream));
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  E.have_S = true;
  E.rec_dirty = true;
  return B200RT_OK;
}

int b200rt_last_residual(b200rt_ctx *c, int e, double *r) {
  if (!c || !r) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_forward(c, b200rt_last_residual(group_owner(c, e), e, r)));
  if (c->mult.defined) { *r = c->mult.residual; return e == 0 ? B200RT_OK : B200RT_ERR_ARG; }
  if (e < 0 || e >= c->n_em) return B200RT_ERR_ARG;
  *r = c->em[e].residual;
  return B200RT_OK;
}

int b200rt_influence_dev(b200rt_ctx *c, int e, void **K, void **S0, void **tsp, void **tab) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_forward(c, b200rt_influence_dev(group_owner_K(c, e), e, K, S0, tsp, tab)));
  if (c->mult.defined) {
    if (e != 0) return B200RT_ERR_ARG;
    Multiplet &M = c->mult;
    if (K) *K = M.K.p;
    if (S0) *S0 = M.S0.p;
    if (tsp) *tsp = M.tau_sp.p;
    if (tab) *tab = M.tau_abs.p;
    M.have_K = true;
    return B200RT_OK;
  }
  if (e < 0 || e >= c->n_em) return B200RT_ERR_ARG;
  Emission &E = c->em[e];
  if (!E.defined) return fail(c, B200RT_ERR_STATE, "emission not defined");
  if (K) *K = E.K.p;
  if (S0) *S0 = E.S0.p;
  if (tsp) *tsp = E.tau_sp.p;
  if (tab) *tab = E.tau_abs.p;
  E.have_K = true;   // the caller may fill rows from peers
  return B200RT_OK;
}

// ---- peer-memory row exchange (one process per GPU): the solving rank exports its K, the others open it and
// name it as the sink of their row batches
int b200rt_ipc_export_influence(b200rt_ctx *c, int e, void *handle64) {
  if (c && c->group) return group_forward(c, b200rt_ipc_export_influence(group_owner_K(c, e), e, handle64));
  if (!c || !handle64 || e < 0 || e >= c->n_em || c->mult.defined) return B200RT_ERR_ARG;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  cudaSetDevice(c->device);
  cudaIpcMemHandle_t h;
  B200RT_CUDA(c, cudaIpcGetMemHandle(&h, c->em[e].K.p));
  std::memcpy(handle64, &h, sizeof h);
  c->em[e].have_K = true;   // peers fill rows
  return B200RT_OK;
}
int b200rt_ipc_open(b200rt_ctx *c, const void *handle64, void **peer_ptr) {
  if (!c || !handle64 || !peer_ptr) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_forward(c, b200rt_ipc_open(group_primary(c), handle64, peer_ptr)));
  cudaSetDevice(c->device);
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle64, sizeof h);
  B200RT_CUDA(c, cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return B200RT_OK;
}
int b200rt_ipc_close(b200rt_ctx *c, void *peer_ptr) {
  if (!c || !peer_ptr) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_forward(c, b200rt_ipc_close(group_primary(c), peer_ptr)));
  cudaSetDevice(c->device);
  for (auto &sk : c->row_sink) if (sk == peer_ptr) sk = nullptr;
  B200RT_CUDA(c, cudaIpcCloseMemHandle(peer_ptr));
  return B200RT_OK;
}
int b200rt_set_row_sink(b200rt_ctx *c, int e, void *peer_K_dev) {
  if (!c || e < 0 || e >= 2) return B200RT_ERR_ARG;
  if (c->group) return fail(c, B200RT_ERR_STATE, "b200rt_set_row_sink: a device group wires its own row sinks");
  if (peer_K_dev) {
    if (c->mult.defined) return fail(c, B200RT_ERR_STATE, "b200rt_set_row_sink: singlet emissions only");
    if (!c->have_grid || e >= c->n_em) return fail(c, B200RT_ERR_STATE, "b200rt_set_row_sink: set the grid and the emissions first");
  }
  c->row_sink[e] = peer_K_dev;
  c->row_sink_n_vox[e] = peer_K_dev ? c->hg.n_vox : 0;
  return B200RT_OK;
}

int b200rt_solve_exchange(b200rt_ctx *c, void **block_dev, void *ipc_handle64) {
  if (!c) return B200RT_ERR_ARG;
  if (c->group) return fail(c, B200RT_ERR_STATE, "b200rt_solve_exchange: a device group wires its own exchange blocks");
  cudaSetDevice(c->device);
  void *p = nullptr;
  if (int rc = api::exchange_block(c, &p)) return rc;
  if (block_dev) *block_dev = p;
  if (ipc_handle64) {
    cudaIpcMemHandle_t h;
    B200RT_CUDA(c, cudaIpcGetMemHandle(&h, p));
    std::memcpy(ipc_handle64, &h, sizeof h);
  }
  return B200RT_OK;
}
int b200rt_solve_distributed(b200rt_ctx *c, int rank, int world, void *const *blocks) {
  if (!c) return B200RT_ERR_ARG;
  if (c->group) return fail(c, B200RT_ERR_STATE, "b200rt_solve_distributed: a device group does this behind b200rt_solve");
  if (!c->have_grid || (c->n_em < 1 && !c->mult.defined)) return fail(c, B200RT_ERR_STATE, "grid / emissions not set");
  cudaSetDevice(c->device);
  return api::solve_distributed(c, rank, world, blocks, true);
}
int b200rt_solve_adjoint(b200rt_ctx *c, int i_emission, int n_rhs, const double *rhs, double *lambda, int *n_steps,
                         double *residual) {
  if (!c) return B200RT_ERR_ARG;
  if (n_rhs < 1 || !rhs || !lambda) return fail(c, B200RT_ERR_ARG, "b200rt_solve_adjoint: n_rhs < 1, or rhs / lambda NULL");
  GROUP_DISPATCH(c, group_solve_adjoint(c, i_emission, n_rhs, rhs, lambda, n_steps, residual));
  if (!c->have_grid || (c->n_em < 1 && !c->mult.defined)) return fail(c, B200RT_ERR_STATE, "grid / emissions not set");
  cudaSetDevice(c->device);
  return api::solve_adjoint(c, i_emission, n_rhs, rhs, lambda, n_steps, residual, false);
}
int b200rt_last_solve_steps(b200rt_ctx *c, int *n_steps) {
  if (!c || !n_steps) return B200RT_ERR_ARG;
  *n_steps = c->group ? group_primary(c)->kry_last_iters : c->kry_last_iters;
  return B200RT_OK;
}

int b200rt_sourcefn_dev(b200rt_ctx *c, int e, void **S) {
  if (c && c->group) return group_forward(c, b200rt_sourcefn_dev(group_owner(c, e), e, S));
  if (c && S && c->mult.defined && e == 0) { *S = c->mult.S.p; return B200RT_OK; }
  if (!c || e < 0 || e >= c->n_em || !S) return B200RT_ERR_ARG;
  *S = c->em[e].S.p;
  return B200RT_OK;
}

int b200rt_los_from_MSO(int precision, int n, const double *loc, const double *dir, double *x, double *y, double *z,
                        double *r, double *t, double *lx, double *ly, double *lz, double *cost) {
  if (n < 0 || !loc || !dir || !x || !y || !z || !r || !t || !lx || !ly || !lz || !cost) return B200RT_ERR_ARG;
  if (precision == B200RT_F64) los_from_MSO<double>(n, loc, dir, x, y, z, r, t, lx, ly, lz, cost);
  else los_from_MSO<float>(n, loc, dir, x, y, z, r, t, lx, ly, lz, cost);
  return B200RT_OK;
}

int b200rt_los_upload(b200rt_ctx *c, int n, const double *x, const double *y, const double *z, const double *r,
                      const double *t, const double *lx, const double *ly, const double *lz, const double *cost) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_los_upload(c, n, x, y, z, r, t, lx, ly, lz, cost));
  if (n <= 0) return fail(c, B200RT_ERR_ARG, "there must be at least one observation to simulate");
  const double *src[9] = {x, y, z, r, t, lx, ly, lz, cost};
  for (auto p : src) if (!p) return fail(c, B200RT_ERR_ARG, "null line-of-sight array");
  cudaSetDevice(c->device);
  return api::los_upload(c, n, src);
}

int b200rt_brightness_resident(b200rt_ctx *c, int n_subsamples) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_brightness_resident(c, n_subsamples));
  if (!c->have_grid || (c->n_em < 1 && !c->mult.defined)) return fail(c, B200RT_ERR_STATE, "grid / emissions not set");
  cudaSetDevice(c->device);
  if (c->mult.defined) return api::mult_brightness(c, n_subsamples);
  return api::brightness_resident(c, n_subsamples);
}

int b200rt_los_download(b200rt_ctx *c, double *B, double *tsp, double *tab, double *col) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_los_download(c, B, tsp, tab, col));
  double *dst[4] = {B, tsp, tab, col};
  return los_download_slice(c, dst, c->n_los, 0);
}

int b200rt_brightness(b200rt_ctx *c, int n, const double *x, const double *y, const double *z, const double *r,
                      const double *t, const double *lx, const double *ly, const double *lz, const double *cost,
                      int n_subsamples, double *B, double *tsp, double *tab, double *col) {
  if (!c) return B200RT_ERR_ARG;
  const double *src[9] = {x, y, z, r, t, lx, ly, lz, cost};
  double *dst[4] = {B, tsp, tab, col};
  GROUP_DISPATCH(c, group_brightness(c, n, src, n_subsamples, dst));
  return brightness_slice(c, n, src, n_subsamples, dst, n, 0);
}

int b200rt_los_weights(b200rt_ctx *c, int n_subsamples, long long *nnz) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_los_weights(c, n_subsamples, nnz));
  cudaSetDevice(c->device);
  return api::los_weights(c, n_subsamples, nnz);
}

int b200rt_los_weights_download(b200rt_ctx *c, long long *row_ptr, int *col, double *val) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_los_weights_download(c, row_ptr, col, val));
  cudaSetDevice(c->device);
  return api::los_weights_download(c, row_ptr, 0, col, val, c->lw.nnz);
}

int b200rt_los_weights_apply(b200rt_ctx *c, int i_emission, int transpose, const double *x, double *y) {
  if (!c || !x || !y || (transpose != 0 && transpose != 1)) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_los_weights_apply(c, i_emission, transpose, x, y));
  cudaSetDevice(c->device);
  return api::los_weights_apply(c, i_emission, transpose, x, y);
}

int b200rt_traverse_voxel_rays(b200rt_ctx *c, int v_begin, int v_end, long long capacity, int *len, int *eb,
                               int *entering, double *distance, long long *n_entries) {
  if (!c || !len || !eb || !entering || !distance) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_forward(c, b200rt_traverse_voxel_rays(group_primary(c), v_begin, v_end, capacity, len, eb, entering, distance, n_entries)));
  if (!c->have_grid) return fail(c, B200RT_ERR_STATE, "grid not set");
  if (v_begin < 0 || v_end > c->hg.n_vox || v_begin > v_end) return fail(c, B200RT_ERR_ARG, "bad voxel range");
  cudaSetDevice(c->device);
  return api::traverse_voxel_rays(c, v_begin, v_end, capacity, len, eb, entering, distance, n_entries);
}

int b200rt_traverse_los(b200rt_ctx *c, long long capacity, int *len, int *eb, int *entering, double *distance,
                        long long *n_entries) {
  if (!c || !len || !eb || !entering || !distance) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_traverse_los(c, capacity, len, eb, entering, distance, n_entries));
  if (!c->have_grid) return fail(c, B200RT_ERR_STATE, "grid not set");
  cudaSetDevice(c->device);
  return api::traverse_los(c, capacity, len, eb, entering, distance, n_entries);
}

int b200rt_last_kernel_ms(b200rt_ctx *c, int phase, float *ms, int *n_launches) {
  if (!c || phase < 0 || phase >= PH_COUNT) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_kernel_ms(c, phase, ms, n_launches));
  if (ms) *ms = c->phase_ms[phase];
  if (n_launches) *n_launches = c->phase_launches[phase];
  return B200RT_OK;
}

int b200rt_iph_load_table(b200rt_ctx *c, const char *fname) {
  if (!c || !fname) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_iph_load_table(c, fname));
  cudaSetDevice(c->device);
  return iph_load_table(c, fname);
}

int b200rt_iph_set_table(b200rt_ctx *c, int kmax, int lmax, int ninf, float temp, const float *alt_au, const float *ang,
                         const float *dans, const float *sot, const float *so, const float *sn, const float *dinf_cm3) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_iph_set_table(c, kmax, lmax, ninf, temp, alt_au, ang, dans, sot, so, sn, dinf_cm3));
  cudaSetDevice(c->device);
  return iph_set_table(c, kmax, lmax, ninf, temp, alt_au, ang, dans, sot, so, sn, dinf_cm3);
}

int b200rt_iph_background(b200rt_ctx *c, float fs, float xpos, float ypos, float zpos, int n_los, const float *u,
                          const float *v, const float *w, float *fln, int *n_steps) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_iph_background(c, fs, xpos, ypos, zpos, n_los, u, v, w, fln, n_steps));
  cudaSetDevice(c->device);
  return iph_background(c, fs, xpos, ypos, zpos, n_los, u, v, w, fln, n_steps);
}

int b200rt_iph_model(b200rt_ctx *c, double g_lya, const double *marspos, int n_los, const double *ra, const double *dec,
                     double *iph_kR) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_iph_model(c, g_lya, marspos, n_los, ra, dec, iph_kR));
  cudaSetDevice(c->device);
  return iph_model(c, g_lya, marspos, n_los, ra, dec, iph_kR);
}

int b200rt_iph_extinction(int n, const double *iph, const double *tau_abs, double *out) {
  if (n < 0 || !iph || !tau_abs || !out) return B200RT_ERR_ARG;
  for (int i = 0; i < n; i++) out[i] = (tau_abs[i] != -1) ? iph[i] * std::exp(-tau_abs[i]) : 0.0;
  return B200RT_OK;
}

int b200rt_measure_fp64_peaks(b200rt_ctx *c, double *dfma, double *dmma) {
  if (!c) return B200RT_ERR_ARG;
  GROUP_DISPATCH(c, group_forward(c, b200rt_measure_fp64_peaks(group_primary(c), dfma, dmma)));
  cudaSetDevice(c->device);
  return measure_fp64_peaks(c, dfma, dmma);
}

} // extern "C"
