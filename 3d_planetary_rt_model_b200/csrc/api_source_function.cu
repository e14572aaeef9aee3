// api_source_function.cu -- influence build with row sinks, single scattering, dense solve, singlet emission tables
// (one of the translation units behind the C ABI; see api_internal.hpp)
#include "api_internal.hpp"

namespace b200rt {
namespace api {
namespace {

// ------------------------------------------------------------------ influence
// ranges: the source-voxel ranges [begin, end) this call builds rows for (one range for a single GPU or a contiguous
// shard; several for the interleaved shards that balance the cost of low- and high-altitude rows across ranks)
template <class Real>
int influence_impl(b200rt_ctx *c, const std::vector<std::pair<int, int>> &ranges) {
  GridView<Real> &g = gv<Real>(c);
  const GridView<Real> &gm = march_gv<Real>(c);   // voxel-origin rays: mirror pairs folded
  const int n_vox = g.n_vox;
  PhaseTimer::reset(c);
  SideStreamDrain drain(c);        // row pushes into a peer's K never outlive the call
  B200RT_CUDA(c, cudaMemsetAsync(c->work_counter.p, 0, 2 * sizeof(int), c->stream));
  B200RT_CUDA(c, cudaMemsetAsync(c->step_counter.p, 0, sizeof(unsigned long long), c->stream));
  int n_rows = 0;
  for (auto &r : ranges) n_rows += r.second - r.first;
  for (int e = 0; e < c->n_em; e++) {
    Emission &E = c->em[e];
    if (!E.defined) return fail(c, B200RT_ERR_STATE, "emission not defined");
    for (auto &r : ranges)
      if (r.second > r.first)
        B200RT_CUDA(c, cudaMemsetAsync(E.K.as<double>() + (size_t) r.first * n_vox, 0,
                                       (size_t) (r.second - r.first) * n_vox * sizeof(double), c->stream));
  }
  // Local slots 0 .. n_rows-1 run over the ranges in order.  One range: slot i is voxel first + i.  Several ranges
  // (interleaved multi-GPU shards): the slot -> voxel map goes to the device, so that a batch -- one traversal launch
  // + one march launch -- spans shard boundaries and the launch count does not grow with the number of shards.
  const bool mapped = ranges.size() > 1;
  std::vector<int> vox_of;
  if (mapped) {
    vox_of.reserve(n_rows);
    for (auto &r : ranges) for (int v = r.first; v < r.second; v++) vox_of.push_back(v);
    B200RT_CUDA(c, c->vox_map.ensure((size_t) n_rows * sizeof(int)));
    B200RT_CUDA(c, cudaMemcpyAsync(c->vox_map.p, vox_of.data(), (size_t) n_rows * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  }
  const int first_voxel = ranges.empty() ? 0 : ranges[0].first;
  const long long cap_rays = batch_capacity(c, sizeof(Real));
  int vox_per_batch = (int) std::max<long long>(1, std::min<long long>(cap_rays / gm.n_rays, std::max(n_rows, 1)));
  bool pushing = false;
  for (int e = 0; e < c->n_em; e++) {
    if (c->row_sink[e] && c->row_sink_n_vox[e] != n_vox)
      return fail(c, B200RT_ERR_STATE, "row sink was named for a different grid (b200rt_set_row_sink after the grid is set)");
    pushing = pushing || c->row_sink[e] != nullptr;
  }
  if (pushing && n_rows > 0) {     // several batches, so that the DMA of one overlaps the march of the next
    if (const char *env = getenv("B200RT_ROW_PUSH_BATCHES")) c->row_push_batches = std::max(1, atoi(env));
    vox_per_batch = std::max(1, std::min(vox_per_batch, (n_rows + c->row_push_batches - 1) / c->row_push_batches));
    if (!c->copy_stream) B200RT_CUDA(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    if (!c->ev_rows) B200RT_CUDA(c, cudaEventCreateWithFlags(&c->ev_rows, cudaEventDisableTiming));
  }
  ListView<Real> lv;
  const long long need = std::max<long long>((long long) vox_per_batch * gm.n_rays, n_vox);
  if (int rc = ensure_lists<Real>(c, need, &lv)) return rc;
  int *overflow = c->work_counter.as<int>() + 1;

  for (int lb = 0; lb < n_rows; lb += vox_per_batch) {
    const int le = std::min(n_rows, lb + vox_per_batch);
    GridView<Real> gb = gm;
    int vb = first_voxel + lb, ve = first_voxel + le;      // unmapped: the voxel range itself
    if (mapped) { gb.vox_map = c->vox_map.as<int>() + lb; vb = 0; ve = le - lb; }
    {
      PhaseTimer t(c, PH_TRAVERSE);
      B200RT_CUDA(c, launch_traverse_voxel_rays<Real>(gb, vb, ve, lv, overflow, c->stream));
      t.stop(1);
      DBG(c, "traverse_voxel_rays");
    }
    for (int e = 0; e < c->n_em; e++) {
      PhaseTimer t(c, PH_INFLUENCE);
      B200RT_CUDA(c, launch_influence<Real>(gb, em_view<Real>(c, e), vb, ve, lv, c->em[e].K.as<double>(),
                                            c->work_counter.as<int>(),
                                            e == 0 ? c->step_counter.as<unsigned long long>() : nullptr, c->stream));
      t.stop(1);
      DBG(c, "influence march");
    }
    if (pushing) {   // the rows of this batch are final: hand them to the solving GPU (peer memory, copy engine, NVLink)
      B200RT_CUDA(c, cudaEventRecord(c->ev_rows, c->stream));
      B200RT_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->ev_rows, 0));
      int run_lo = lb;                                      // contiguous runs of voxels inside the batch
      while (run_lo < le) {
        int run_hi = run_lo + 1;
        const int v_lo = mapped ? vox_of[run_lo] : first_voxel + run_lo;
        while (run_hi < le && (mapped ? vox_of[run_hi] : first_voxel + run_hi) == v_lo + (run_hi - run_lo)) run_hi++;
        for (int e = 0; e < c->n_em; e++)
          if (c->row_sink[e])
            B200RT_CUDA(c, cudaMemcpyAsync(static_cast<double *>(c->row_sink[e]) + (size_t) v_lo * n_vox,
                                           c->em[e].K.as<double>() + (size_t) v_lo * n_vox,
                                           (size_t) (run_hi - run_lo) * n_vox * sizeof(double), cudaMemcpyDeviceToDevice,
                                           c->copy_stream));
        run_lo = run_hi;
      }
    }
  }
  // single scattering: one sun-ward ray per voxel (every rank computes all of them: n_vox rays)
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
      DBG(c, "traverse sun rays");
    }
    for (int e = 0; e < c->n_em; e++) {
      PhaseTimer t(c, PH_INFLUENCE);
      Emission &E = c->em[e];
      B200RT_CUDA(c, launch_single_scattering<Real>(g, em_view<Real>(c, e), lv, shadow, E.S0.as<double>(),
                                                    E.tau_sp.as<double>(), E.tau_abs.as<double>(),
                                                    c->work_counter.as<int>(), c->stream));
      t.stop(1);
      DBG(c, "single scattering march");
    }
  }
  B200RT_CUDA(c, c->host_words.ensure(4 * sizeof(unsigned long long)));
  unsigned long long *steps_p = c->host_words.as<unsigned long long>() + 1;
  B200RT_CUDA(c, cudaMemcpyAsync(steps_p, c->step_counter.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  const int rc_overflow = check_overflow(c);   // synchronises
  const unsigned long long steps = *steps_p;
  if (pushing) B200RT_CUDA(c, cudaStreamSynchronize(c->copy_stream));   // the rows have landed on the solving GPU
  if (rc_overflow) return rc_overflow;
  PhaseTimer::collect(c);
  c->last_steps = (long long) steps;
  for (int e = 0; e < c->n_em; e++) { c->em[e].have_K = true; c->em[e].have_S = false; }
  c->built_ranges = ranges;
  return B200RT_OK;
}

// only_e >= 0: that emission alone (a device group solves emission e on the device that gathered its rows)
int solve_impl(b200rt_ctx *c, bool reset_timer, int only_e = -1) {
  const int n = c->hg.n_vox;
  // Large systems whose rows were all built here: preconditioned GMRES (solve_krylov.cu with one rank: 4.0 ms against the
  // LU's 5.8 ms at n = 5841, S within 1e-11 of the LU's element by element).  The LU below stays the solve of small
  // systems (a 741-unknown LU is 0.4 ms, shorter than the iteration's set-up), of matrices assembled from peers' row
  // pushes, and the fallback when the iteration does not converge.  B200RT_SOLVER = lu | gmres overrides the size rule.
  if (only_e < 0) {
    bool have_all = true;
    for (int e = 0; e < c->n_em; e++) have_all = have_all && c->em[e].have_K;
    if (have_all && use_gmres(c) && n <= B200RT_KRYLOV_MAX_N) {
      void *block = nullptr;
      if (int rc = exchange_block(c, &block)) return rc;
      const int rc = solve_distributed(c, 0, 1, &block, reset_timer);
      if (rc != B200RT_ERR_NOT_DOMINANT) return rc;
      // not converged: the direct solve decides (and reports a matrix it cannot take)
    }
  }
  if (reset_timer) PhaseTimer::reset(c);
  for (int e = 0; e < c->n_em; e++) {
    if (only_e >= 0 && e != only_e) continue;
    Emission &E = c->em[e];
    if (!E.have_K) return fail(c, B200RT_ERR_STATE, "b200rt_solve: influence matrix not built");
    PhaseTimer t(c, PH_SOLVE);
    SolveResult r = {0, 0, 0};
    if (int rc = solve_dense(c, n, E.K.as<double>(), E.branching, E.S0.as<double>(), E.S.as<double>(), &r)) return rc;
    t.stop(r.launches);
    E.residual = r.residual;
    if (c->precision == B200RT_F64)
      B200RT_CUDA(c, launch_convert<double>(E.S.as<double>(), E.S_real.as<double>(), n, c->stream));
    else
      B200RT_CUDA(c, launch_convert<float>(E.S.as<double>(), E.S_real.as<float>(), n, c->stream));
    E.have_S = true;
    E.rec_dirty = true;
  }
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  PhaseTimer::collect(c);
  return B200RT_OK;
}

template <class Real>
int set_singlet_impl(b200rt_ctx *c, int e, const double *const arr[8]) {
  const int n = c->hg.n_vox;
  Emission &E = c->em[e];
  B200RT_CUDA(c, E.tabs.ensure((size_t) 8 * n * sizeof(Real)));
  B200RT_CUDA(c, E.phi.ensure((size_t) n * N_LAMBDA * sizeof(Real)));
  B200RT_CUDA(c, E.mrec.ensure((size_t) n * 2 * N_LAMBDA * sizeof(Real)));
  B200RT_CUDA(c, E.K.ensure((size_t) n * n * sizeof(double)));
  B200RT_CUDA(c, E.S0.ensure(n * sizeof(double)));
  B200RT_CUDA(c, E.tau_sp.ensure(n * sizeof(double)));
  B200RT_CUDA(c, E.tau_abs.ensure(n * sizeof(double)));
  B200RT_CUDA(c, E.S.ensure(n * sizeof(double)));
  B200RT_CUDA(c, E.S_real.ensure(n * sizeof(Real)));
  B200RT_CUDA(c, E.rec_pt.ensure((size_t) n * 8 * sizeof(Real)));
  B200RT_CUDA(c, E.rec_avg.ensure((size_t) n * 8 * sizeof(Real)));
  E.rec_dirty = true;
  // the eight tables travel as ONE truly asynchronous copy out of page-locked staging (eight copies out of the caller's
  // pageable arrays would each be staged by the runtime under a process-wide lock: with many contexts -- the sweep's 8-32
  // worker threads -- that lock, not the GPUs, set the rate)
  const size_t bytes = (size_t) 8 * n * sizeof(double);
  B200RT_CUDA(c, c->host_stage.ensure(bytes));
  for (int a = 0; a < 8; a++) std::memcpy(c->host_stage.as<double>() + (size_t) a * n, arr[a], (size_t) n * sizeof(double));
  if (sizeof(Real) == sizeof(double)) {
    B200RT_CUDA(c, cudaMemcpyAsync(E.tabs.p, c->host_stage.p, bytes, cudaMemcpyHostToDevice, c->stream));
  } else {
    B200RT_CUDA(c, c->dev_stage.ensure(bytes));
    B200RT_CUDA(c, cudaMemcpyAsync(c->dev_stage.p, c->host_stage.p, bytes, cudaMemcpyHostToDevice, c->stream));
    B200RT_CUDA(c, launch_convert<Real>(c->dev_stage.as<double>(), E.tabs.as<Real>(), (long long) 8 * n, c->stream));
  }
  B200RT_CUDA(c, launch_phi_table<Real>(E.tabs.as<Real>(), E.tabs.as<Real>() + 2 * (size_t) n, E.tabs.as<Real>() + 3 * (size_t) n, n,
                                        E.phi.as<Real>(), E.mrec.as<Real>(), c->stream));
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  return B200RT_OK;
}


}  // namespace

bool use_gmres(const b200rt_ctx *c) {
  const long long n_vox = c->hg.n_vox;
  long long min_n = 2048;
  if (const char *env = getenv("B200RT_KRYLOV_MIN_N")) min_n = atoll(env);
  bool iterate = n_vox >= min_n;
  if (const char *env = getenv("B200RT_SOLVER")) iterate = std::strcmp(env, "gmres") == 0 || (iterate && std::strcmp(env, "lu") != 0);
  long long own = 0;
  for (auto &r : c->built_ranges) own += r.second - r.first;
  return iterate && own == n_vox;
}

int influence(b200rt_ctx *c, const std::vector<std::pair<int, int>> &ranges) {
  return is64(c) ? influence_impl<double>(c, ranges) : influence_impl<float>(c, ranges);
}
int solve(b200rt_ctx *c, bool reset_timer) { return solve_impl(c, reset_timer); }
int solve_emission(b200rt_ctx *c, int e) {
  if (e < 0 || e >= c->n_em) return fail(c, B200RT_ERR_ARG, "bad emission index");
  cudaSetDevice(c->device);
  return solve_impl(c, true, e);
}
int set_singlet(b200rt_ctx *c, int e, const double *const arr[8]) {
  return is64(c) ? set_singlet_impl<double>(c, e, arr) : set_singlet_impl<float>(c, e, arr);
}

}  // namespace api
}  // namespace b200rt
