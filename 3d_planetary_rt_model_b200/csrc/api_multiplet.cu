// api_multiplet.cu -- the multiplet CFR emissions: tables, influence build, solve, brightness, download
// (one of the translation units behind the C ABI; see api_internal.hpp)
#include "api_internal.hpp"

namespace b200rt {
namespace api {
namespace {

// ------------------------------------------------------------------ multiplet emission
template <class Real>
MultView<Real> mult_view(b200rt_ctx *c) {
  Multiplet &M = c->mult;
  const size_t n = c->hg.n_vox;
  Real *t = M.tabs.as<Real>();
  MultView<Real> v;
  v.T = t; v.T_pt = t + n; v.nabs = t + 2 * n; v.nabs_pt = t + 3 * n;
  for (int l = 0; l < MULT_MAX_LOWER; l++) { v.n[l] = t + (4 + l) * n; v.n_pt[l] = t + (7 + l) * n; }
  v.rec_step = M.rec_step.as<Real>(); v.rec_org = M.rec_org.as<Real>(); v.rec_w0 = M.rec_w0.as<Real>();
  v.tsv = M.tsv.as<Real>(); v.tav = M.tav.as<Real>();
  v.S = M.S_real.as<Real>();
  v.rec_pt = M.rec_pt.as<Real>(); v.rec_avg = M.rec_avg.as<Real>();
  return v;
}

template <class Real>
int set_multiplet_impl(b200rt_ctx *c, const double *const arr[6]) {
  Multiplet &M = c->mult;
  const b200rt_multiplet_desc &d = M.d;
  const size_t n = c->hg.n_vox, ne = n * d.n_upper;
  const size_t nlp = (d.n_lambda + MULT_LPR - 1) / MULT_LPR, slots = n * MULT_LPR * nlp;
  B200RT_CUDA(c, M.tabs.ensure(10 * n * sizeof(Real)));
  B200RT_CUDA(c, cudaMemsetAsync(M.tabs.p, 0, 10 * n * sizeof(Real), c->stream));
  B200RT_CUDA(c, M.rec_step.ensure(slots * (d.n_multiplets + d.n_lines) * sizeof(Real)));
  B200RT_CUDA(c, M.rec_org.ensure(slots * d.n_lines * sizeof(Real)));
  B200RT_CUDA(c, M.rec_w0.ensure(slots * d.n_lines * sizeof(Real)));
  B200RT_CUDA(c, M.tsv.ensure(n * d.n_lines * sizeof(Real)));
  B200RT_CUDA(c, M.tav.ensure(n * d.n_lines * sizeof(Real)));
  B200RT_CUDA(c, M.K.ensure(ne * ne * sizeof(double)));
  B200RT_CUDA(c, M.S0.ensure(ne * sizeof(double)));
  B200RT_CUDA(c, M.S.ensure(ne * sizeof(double)));
  B200RT_CUDA(c, M.S_real.ensure(ne * sizeof(Real)));
  B200RT_CUDA(c, M.tau_sp.ensure(n * d.n_lines * sizeof(double)));
  B200RT_CUDA(c, M.tau_abs.ensure(n * d.n_lines * sizeof(double)));
  B200RT_CUDA(c, M.rec_pt.ensure(n * MULT_REC * sizeof(Real)));
  B200RT_CUDA(c, M.rec_avg.ensure(n * MULT_REC * sizeof(Real)));
  Real *t = M.tabs.as<Real>();
  DevBuf stage;
  int rc = B200RT_OK;
  // arr: species_density [n_lower][n], species_density_pt, T, T_pt, absorber, absorber_pt
  for (int l = 0; l < d.n_lower && rc == B200RT_OK; l++) {
    rc = upload_real<Real>(c, arr[0] + (size_t) l * n, t + (4 + l) * n, n, stage);
    if (rc == B200RT_OK) rc = upload_real<Real>(c, arr[1] + (size_t) l * n, t + (7 + l) * n, n, stage);
  }
  for (int a = 0; a < 4 && rc == B200RT_OK; a++) rc = upload_real<Real>(c, arr[2 + a], t + (size_t) a * n, n, stage);
  if (rc == B200RT_OK) {
    cudaError_t er = launch_mult_tables<Real>(d, mult_view<Real>(c), (int) n, c->stream);
    if (er == cudaSuccess) er = cudaStreamSynchronize(c->stream);
    if (er != cudaSuccess) rc = fail(c, B200RT_ERR_CUDA, cudaGetErrorString(er));
  }
  stage.release();
  return rc;
}

// ranges: the source-voxel ranges [begin, end) this call builds the rows of (all n_upper element rows of each voxel);
// several ranges are the interleaved shards of a distributed solve, marched as one list as in influence_impl
template <class Real>
int mult_influence_impl(b200rt_ctx *c, const std::vector<std::pair<int, int>> &ranges) {
  GridView<Real> &g = gv<Real>(c);
  const GridView<Real> &gm = march_gv<Real>(c);   // voxel-origin rays: mirror pairs folded
  Multiplet &M = c->mult;
  const b200rt_multiplet_desc &d = M.d;
  const int n_vox = g.n_vox;
  const size_t ne = (size_t) n_vox * d.n_upper;
  PhaseTimer::reset(c);
  B200RT_CUDA(c, cudaMemsetAsync(c->work_counter.p, 0, 2 * sizeof(int), c->stream));
  B200RT_CUDA(c, cudaMemsetAsync(c->step_counter.p, 0, sizeof(unsigned long long), c->stream));
  int n_rows = 0;
  for (auto &r : ranges) {
    n_rows += r.second - r.first;
    if (r.second > r.first)
      B200RT_CUDA(c, cudaMemsetAsync(M.K.as<double>() + (size_t) r.first * d.n_upper * ne, 0,
                                     (size_t) (r.second - r.first) * d.n_upper * ne * sizeof(double), c->stream));
  }
  const bool mapped = ranges.size() > 1;
  if (mapped) {
    std::vector<int> vox_of;
    vox_of.reserve(n_rows);
    for (auto &r : ranges) for (int v = r.first; v < r.second; v++) vox_of.push_back(v);
    B200RT_CUDA(c, c->vox_map.ensure((size_t) n_rows * sizeof(int)));
    B200RT_CUDA(c, cudaMemcpyAsync(c->vox_map.p, vox_of.data(), (size_t) n_rows * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    B200RT_CUDA(c, cudaStreamSynchronize(c->stream));   // (vox_of is pageable and goes out of scope)
  }
  const int first_voxel = ranges.empty() ? 0 : ranges[0].first;
  const long long cap_rays = batch_capacity(c, sizeof(Real));
  const int vox_per_batch = (int) std::max<long long>(1, std::min<long long>(cap_rays / gm.n_rays, n_rows));
  ListView<Real> lv;
  const long long need = std::max<long long>((long long) vox_per_batch * gm.n_rays, n_vox);
  if (int rc = ensure_lists<Real>(c, need, &lv)) return rc;
  int *overflow = c->work_counter.as<int>() + 1;
  MultView<Real> mv = mult_view<Real>(c);
  for (int lb = 0; lb < n_rows; lb += vox_per_batch) {
    const int le = std::min(n_rows, lb + vox_per_batch);
    GridView<Real> gb = gm;
    int vb = first_voxel + lb, ve = first_voxel + le;      // unmapped: the voxel range itself
    if (mapped) { gb.vox_map = c->vox_map.as<int>() + lb; vb = 0; ve = le - lb; }
    {
      PhaseTimer t(c, PH_TRAVERSE);
      B200RT_CUDA(c, launch_traverse_voxel_rays<Real>(gb, vb, ve, lv, overflow, c->stream));
      t.stop(1);
    }
    {
      PhaseTimer t(c, PH_INFLUENCE);
      B200RT_CUDA(c, launch_mult_influence<Real>(d, gb, mv, vb, ve, lv, M.K.as<double>(), c->work_counter.as<int>(),
                                                 c->step_counter.as<unsigned long long>(), c->stream));
      t.stop(1);
      DBG(c, "multiplet influence march");
    }
  }
  {
    const Real *sp = c->sun_rays.as<Real>();
    RayList<Real> rl;
    rl.r = sp + 0 * (size_t) n_vox; rl.z = sp + 1 * (size_t) n_vox; rl.t = sp + 2 * (size_t) n_vox;
    rl.cost = sp + 3 * (size_t) n_vox; rl.lz = sp + 4 * (size_t) n_vox;
    const int *ip = reinterpret_cast<const int *>(sp + 5 * (size_t) n_vox);
    rl.i_voxel = ip;
    const int *shadow = ip + n_vox;
    {
      PhaseTimer t(c, PH_TRAVERSE);
      B200RT_CUDA(c, launch_traverse_list<Real>(g, rl, n_vox, lv, overflow, c->stream));
      t.stop(1);
    }
    {
      PhaseTimer t(c, PH_INFLUENCE);
      B200RT_CUDA(c, cudaMemsetAsync(M.S0.p, 0, ne * sizeof(double), c->stream));
      B200RT_CUDA(c, launch_mult_single_scattering<Real>(d, g, mv, lv, shadow, M.S0.as<double>(), M.tau_sp.as<double>(),
                                                         M.tau_abs.as<double>(), c->work_counter.as<int>(), c->stream));
      t.stop(1);
      DBG(c, "multiplet single scattering");
    }
  }
  B200RT_CUDA(c, c->host_words.ensure(4 * sizeof(unsigned long long)));
  unsigned long long *steps_p = c->host_words.as<unsigned long long>() + 1;
  B200RT_CUDA(c, cudaMemcpyAsync(steps_p, c->step_counter.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  if (int rc = check_overflow(c)) return rc;
  const unsigned long long steps = *steps_p;
  PhaseTimer::collect(c);
  c->last_steps = (long long) steps;
  M.have_K = true; M.have_S = false;
  c->built_ranges = ranges;
  return B200RT_OK;
}

int mult_solve_impl(b200rt_ctx *c, bool reset_timer) {
  Multiplet &M = c->mult;
  const int ne = c->hg.n_vox * M.d.n_upper;
  if (!M.have_K) return fail(c, B200RT_ERR_STATE, "b200rt_solve: influence matrix not built");
  // the singlet's rule (api_source_function.cu, solve_impl): grids of B200RT_KRYLOV_MIN_N voxels and more whose rows were
  // all built here take the GMRES over the n_el elements, the LU decides when it does not converge
  if (use_gmres(c) && ne <= B200RT_KRYLOV_MAX_N) {
    void *block = nullptr;
    if (int rc = exchange_block(c, &block)) return rc;
    const int rc = solve_distributed(c, 0, 1, &block, reset_timer);
    if (rc != B200RT_ERR_NOT_DOMINANT) return rc;
  }
  if (reset_timer) PhaseTimer::reset(c);
  PhaseTimer t(c, PH_SOLVE);
  SolveResult r = {0, 0, 0};
  // multiplet_CFR_emission::pre_solve is empty: kernel = I - K (multiplet_CFR_emission.hpp:408; emission_voxels.hpp:170-176)
  if (int rc = solve_dense(c, ne, M.K.as<double>(), 1.0, M.S0.as<double>(), M.S.as<double>(), &r)) return rc;
  t.stop(r.launches);
  M.residual = r.residual;
  if (c->precision == B200RT_F64) B200RT_CUDA(c, launch_convert<double>(M.S.as<double>(), M.S_real.as<double>(), ne, c->stream));
  else B200RT_CUDA(c, launch_convert<float>(M.S.as<double>(), M.S_real.as<float>(), ne, c->stream));
  M.have_S = true;
  M.rec_dirty = true;
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  PhaseTimer::collect(c);
  return B200RT_OK;
}

template <class Real>
int mult_brightness_impl(b200rt_ctx *c, int n_subsamples) {
  Multiplet &M = c->mult;
  const b200rt_multiplet_desc &d = M.d;
  if (n_subsamples == 1 || n_subsamples < 0)
    return fail(c, B200RT_ERR_ARG, "n_subsamples must be 0 or > 1 (RT_grid.hpp:237)");
  if (c->n_los <= 0) return fail(c, B200RT_ERR_STATE, "no lines of sight uploaded");
  if (c->hg.pp)
    return fail(c, B200RT_ERR_STATE, "interp_weights not implemented in grid_plane_parallel (grid_plane_parallel.hpp:304-311)");
  if (!M.have_S) return fail(c, B200RT_ERR_STATE, "source function not available (solve or set_sourcefn first)");
  GridView<Real> &g = gv<Real>(c);
  PhaseTimer::reset(c);
  B200RT_CUDA(c, cudaMemsetAsync(c->work_counter.p, 0, 2 * sizeof(int), c->stream));
  const long long n = c->n_los;
  const long long per_batch = std::min<long long>(batch_capacity(c, sizeof(Real)), n);
  ListView<Real> lv;
  if (int rc = ensure_lists<Real>(c, per_batch, &lv)) return rc;
  const size_t n_out = 3 * d.n_lines + d.n_lower;
  B200RT_CUDA(c, c->los_out.ensure(n_out * n * sizeof(Real)));
  B200RT_CUDA(c, c->los_order.ensure(((size_t) per_batch + 2 * (size_t) (c->hg.cap + 1)) * sizeof(int)));
  const Real *li = c->los_in.as<Real>();
  MultView<Real> mv = mult_view<Real>(c);
  if (M.rec_dirty) {
    B200RT_CUDA(c, launch_mult_pack<Real>(d, mv, g.n_vox, c->stream));
    M.rec_dirty = false;
  }
  int *overflow = c->work_counter.as<int>() + 1;
  for (long long first = 0; first < n; first += per_batch) {
    const long long count = std::min(per_batch, n - first);
    RayList<Real> rl;
    rl.r = li + 3 * n + first; rl.z = li + 2 * n + first; rl.t = li + 4 * n + first;
    rl.cost = li + 8 * n + first; rl.lz = li + 7 * n + first; rl.i_voxel = nullptr;
    {
      PhaseTimer t(c, PH_TRAVERSE);
      B200RT_CUDA(c, launch_traverse_list<Real>(g, rl, count, lv, overflow, c->stream));
      t.stop(1);
    }
    const int *order = nullptr;
    if (lv.cap <= LOS_ORDER_MAX_CAP && count >= los_order_min()) {
      PhaseTimer t(c, PH_ORDER);
      int *bins = c->los_order.as<int>(), *ord = bins + 2 * (lv.cap + 1);
      B200RT_CUDA(c, launch_los_order(lv.len, count, lv.cap, bins, ord, c->stream));
      order = ord;
      t.stop(3);
    }
    {
      PhaseTimer t(c, PH_BRIGHTNESS);
      B200RT_CUDA(c, launch_mult_brightness<Real>(d, g, mv, li, n, first, count, lv, n_subsamples, c->los_out.as<Real>(), n,
                                                  c->work_counter.as<int>(), order, c->stream));
      t.stop(1);
    }
  }
  if (int rc = check_overflow(c)) return rc;
  PhaseTimer::collect(c);
  c->los_done = true;
  return B200RT_OK;
}

// multiplet outputs [3 n_lines + n_lower][n_los] -> brightness, tau_species_final, tau_absorber_final [n_lines][n],
// species_col_dens [n_lower][n]
template <class Real>
int mult_los_download_impl(b200rt_ctx *c, double *const dst[4], long long stride, long long offset) {
  const long long n = c->n_los;
  const b200rt_multiplet_desc &d = c->mult.d;
  const Real *o = c->los_out.as<Real>();
  const int rows[4] = {d.n_lines, d.n_lines, d.n_lines, d.n_lower};
  size_t row0 = 0;
  std::vector<float> tmp;
  for (int q = 0; q < 4; q++) {
    if (dst[q])
      for (int r = 0; r < rows[q]; r++) {
        const Real *src = o + (row0 + r) * (size_t) n;
        double *out = dst[q] + (size_t) r * stride + offset;
        if (sizeof(Real) == sizeof(double)) {
          B200RT_CUDA(c, cudaMemcpyAsync(out, src, (size_t) n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        } else {
          tmp.resize(n);
          B200RT_CUDA(c, cudaMemcpyAsync(tmp.data(), src, (size_t) n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
          B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
          for (long long i = 0; i < n; i++) out[i] = tmp[i];
        }
      }
    row0 += rows[q];
  }
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  return B200RT_OK;
}


}  // namespace

int set_multiplet(b200rt_ctx *c, const double *const arr[6]) {
  return is64(c) ? set_multiplet_impl<double>(c, arr) : set_multiplet_impl<float>(c, arr);
}
int mult_influence(b200rt_ctx *c, const std::vector<std::pair<int, int>> &ranges) {
  return is64(c) ? mult_influence_impl<double>(c, ranges) : mult_influence_impl<float>(c, ranges);
}
int mult_solve(b200rt_ctx *c, bool reset_timer) { return mult_solve_impl(c, reset_timer); }
int mult_brightness(b200rt_ctx *c, int n_subsamples) {
  return is64(c) ? mult_brightness_impl<double>(c, n_subsamples) : mult_brightness_impl<float>(c, n_subsamples);
}
int mult_los_download(b200rt_ctx *c, double *const dst[4], long long stride, long long offset) {
  return is64(c) ? mult_los_download_impl<double>(c, dst, stride, offset) : mult_los_download_impl<float>(c, dst, stride, offset);
}

}  // namespace api
}  // namespace b200rt
