// api_internal.hpp -- what the translation units behind the C ABI share (nothing here is part of include/b200rt.h):
// phase timing, scratch sizing, uploads, and the per-subsystem entry functions that b200rt_api.cu's extern "C" layer calls.
//   b200rt_api.cu            the extern "C" functions: argument checks, device-group dispatch, context lifetime
//   api_source_function.cu   influence build (+ row sinks), single scattering, solve, singlet emission tables
//   api_brightness.cu        line-of-sight upload / brightness (resident and pipelined host-buffer forms) / download
//   api_traverse.cu          the traversal parity surface (boundary lists back to the host)
//   api_multiplet.cu         the same four steps for the multiplet CFR emissions
//   api_weights.cu           line-of-sight weighting functions: build, download, products
#pragma once
#include <algorithm>
#include <cmath>
#include <cstring>
#include <cstdlib>
#include <new>
#include <utility>
#include <vector>
#include "common.hpp"

namespace b200rt {
namespace api {


// Boundary-list scratch per batch: 8 GiB of the 180 GB, so that the bench workload (1e6 lines of sight and 2.24e6 voxel
// rays on the 100x60 grid, 1.12e6 of them marched once mirror pairs are folded: 3.1 and 3.5 GB of lists) runs as ONE
// batch per phase.  Every batch boundary drains the
// persistent brightness kernel (a single line of sight takes ~0.5 ms): measured 1.45 ms per boundary (r01n launch
// list: 686k LOS in 29.63 ms, 314k in 14.35 ms).  B200RT_SCRATCH_BYTES overrides it (tests force several batches).
constexpr size_t SCRATCH_BUDGET_BYTES = size_t(1) << 33;

// Events come from a per-context pool (created once, reused by every call): a parameter-set sweep makes ~25 timers per
// set on each of 8-16 threads, and event creation / destruction goes through process-wide runtime state.
struct PhaseTimer {
  b200rt_ctx *c;
  int phase;
  cudaEvent_t a, b;
  static cudaEvent_t take(b200rt_ctx *c) {
    if (c->timer_used == c->timer_events.size()) {
      cudaEvent_t e = nullptr;
      cudaEventCreate(&e);
      c->timer_events.push_back(e);
    }
    return c->timer_events[c->timer_used++];
  }
  PhaseTimer(b200rt_ctx *ctx, int ph) : c(ctx), phase(ph), a(take(ctx)), b(take(ctx)) { cudaEventRecord(a, c->stream); }
  PhaseTimer(const PhaseTimer &) = delete;
  void stop(int launches) {
    cudaEventRecord(b, c->stream);
    pending().push_back({phase, launches, a, b});
  }
  struct Rec { int phase, launches; cudaEvent_t a, b; };
  static std::vector<Rec> &pending() { static thread_local std::vector<Rec> v; return v; }
  static void reset(b200rt_ctx *c) {
    for (int p = 0; p < PH_COUNT; p++) { c->phase_ms[p] = 0; c->phase_launches[p] = 0; }
    pending().clear();   // records an error path left behind; their events stay in the pool
    c->timer_used = 0;
  }
  static void collect(b200rt_ctx *c) {   // call after the stream has been synchronised
    for (auto &r : pending()) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) c->phase_ms[r.phase] += ms;
      c->phase_launches[r.phase] += r.launches;
    }
    pending().clear();
    c->timer_used = 0;
  }
};

// B200RT_DEBUG_SYNC=1: synchronise after every launch so a fault is attributed to its kernel
inline int dbg_sync(b200rt_ctx *c, const char *what) {
  static const bool on = getenv("B200RT_DEBUG_SYNC") != nullptr;
  if (!on) return B200RT_OK;
  cudaError_t e = cudaStreamSynchronize(c->stream);
  if (e != cudaSuccess) return fail(c, B200RT_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
  return B200RT_OK;
}
#define DBG(c, what) do { if (int rc__ = dbg_sync(c, what)) return rc__; } while (0)

template <class Real>
GridView<Real> &gv(b200rt_ctx *c) { return *static_cast<GridView<Real> *>(c->grid_view); }
// the influence builds march this one: mirror pairs of voxel-origin rays folded (grid_host.cpp, fold_pairs)
template <class Real>
GridView<Real> &march_gv(b200rt_ctx *c) { return *static_cast<GridView<Real> *>(c->march_view); }

template <class Real>
EmissionView<Real> em_view(b200rt_ctx *c, int e) {
  const Emission &E = c->em[e];
  const int n = c->hg.n_vox;
  const Real *t = E.tabs.as<Real>();
  EmissionView<Real> v;
  v.T_ratio = t + 0 * n; v.density = t + 1 * n; v.dtau_species = t + 2 * n; v.dtau_absorber = t + 3 * n;
  v.T_ratio_pt = t + 4 * n; v.density_pt = t + 5 * n; v.dtau_species_pt = t + 6 * n; v.dtau_absorber_pt = t + 7 * n;
  v.phi = E.phi.as<Real>();
  v.mrec = E.mrec.as<Real>();
  v.sourcefn = E.S_real.as<Real>();
  v.rec_pt = E.rec_pt.as<Real>(); v.rec_avg = E.rec_avg.as<Real>();
  v.branching = (Real) E.branching; v.sigma_ref = (Real) E.sigma_ref; v.g_factor = (Real) E.g_factor;
  return v;
}

template <class Real>
int ensure_lists(b200rt_ctx *c, long long n_rays, ListView<Real> *lv) {
  const int cap = c->hg.cap;
  B200RT_CUDA(c, c->list_dist.ensure((size_t) n_rays * cap * sizeof(Real)));
  B200RT_CUDA(c, c->list_ent.ensure((size_t) n_rays * cap * sizeof(int)));
  B200RT_CUDA(c, c->list_len.ensure((size_t) n_rays * sizeof(int)));
  B200RT_CUDA(c, c->list_flag.ensure((size_t) n_rays * sizeof(int)));
  lv->dist = c->list_dist.as<Real>(); lv->ent = c->list_ent.as<int>();
  lv->len = c->list_len.as<int>(); lv->flag = c->list_flag.as<int>(); lv->cap = cap;
  return B200RT_OK;
}

// The longest-first order only pays when the queue is several times deeper than the machine (148 SMs x 4 CTAs x 32
// 4-lane groups = 18944 lines of sight in flight): below that every group gets at most a few lines of sight and the
// order only concentrates the long ones in the first CTAs.  B200RT_LOS_ORDER_MIN overrides (tests, diagnosis).
inline long long los_order_min() {
  if (const char *env = getenv("B200RT_LOS_ORDER_MIN")) return atoll(env);
  return 4LL * NUM_SMS * 4 * 32;
}

inline long long batch_capacity(b200rt_ctx *c, size_t real_bytes) {
  const size_t per_ray = (size_t) c->hg.cap * (real_bytes + sizeof(int)) + 2 * sizeof(int);
  size_t budget = SCRATCH_BUDGET_BYTES;
  if (const char *env = getenv("B200RT_SCRATCH_BYTES")) budget = (size_t) std::max(1LL, atoll(env));
  long long n = (long long) (budget / per_ray);
  return std::max<long long>(n, 1);
}

inline int check_overflow(b200rt_ctx *c) {
  B200RT_CUDA(c, c->host_words.ensure(4 * sizeof(unsigned long long)));
  int *flag_p = c->host_words.as<int>();
  *flag_p = 0;
  B200RT_CUDA(c, cudaMemcpyAsync(flag_p, c->work_counter.as<int>() + 1, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  const int flag = *flag_p;
  if (flag)
    return fail(c, B200RT_ERR_CAPACITY, "a ray crossed more than 2*n_rb+n_sb boundaries (crossing list capacity)");
  return B200RT_OK;
}

// upload a host double array into a device Real array (widening/narrowing on the device)
template <class Real>
int upload_real(b200rt_ctx *c, const double *src, Real *dst, size_t n, DevBuf &stage);
template <>
inline int upload_real<double>(b200rt_ctx *c, const double *src, double *dst, size_t n, DevBuf &) {
  B200RT_CUDA(c, cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  return B200RT_OK;
}
template <>
inline int upload_real<float>(b200rt_ctx *c, const double *src, float *dst, size_t n, DevBuf &stage) {
  B200RT_CUDA(c, stage.ensure(n * sizeof(double)));
  B200RT_CUDA(c, cudaMemcpyAsync(stage.p, src, n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  B200RT_CUDA(c, launch_convert<float>(stage.as<double>(), dst, (long long) n, c->stream));
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));   // stage is reused by the caller
  return B200RT_OK;
}

// leaves nothing in flight on the side streams of a call -- peer row pushes, uploads from / downloads into caller arrays
// -- whichever way the call returns (an early error return included)
struct SideStreamDrain {
  b200rt_ctx *c;
  explicit SideStreamDrain(b200rt_ctx *ctx) : c(ctx) {}
  SideStreamDrain(const SideStreamDrain &) = delete;
  ~SideStreamDrain() {
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    if (c->out_stream) cudaStreamSynchronize(c->out_stream);
  }
};

inline bool is64(const b200rt_ctx *c) { return c->precision == B200RT_F64; }

// ---- api_source_function.cu
int influence(b200rt_ctx *c, const std::vector<std::pair<int, int>> &ranges);
int solve(b200rt_ctx *c, bool reset_timer);
int solve_emission(b200rt_ctx *c, int e);   // one singlet emission only (device group: emission e on its owner device)
// b200rt_solve's choice of the GMRES (solve_krylov.cu) over the LU: a grid of B200RT_KRYLOV_MIN_N voxels or more (default
// 2048) whose rows were all built by this context; B200RT_SOLVER = lu | gmres overrides the size.  The caller adds the
// capacity limit (B200RT_KRYLOV_MAX_N unknowns) and that the rows exist.
bool use_gmres(const b200rt_ctx *c);
int set_singlet(b200rt_ctx *c, int e, const double *const arr[8]);
// ---- api_brightness.cu  (los_download_slice / brightness_slice are declared in common.hpp)
int brightness_resident(b200rt_ctx *c, int n_subsamples);
int los_upload(b200rt_ctx *c, int n, const double *const src[9]);
// ---- api_traverse.cu
int traverse_voxel_rays(b200rt_ctx *c, int v_begin, int v_end, long long capacity, int *len, int *exits_bottom,
                        int *entering, double *distance, long long *n_entries);
int traverse_los(b200rt_ctx *c, long long capacity, int *len, int *exits_bottom, int *entering, double *distance,
                 long long *n_entries);
// ---- api_multiplet.cu
int set_multiplet(b200rt_ctx *c, const double *const arr[6]);
int mult_influence(b200rt_ctx *c, const std::vector<std::pair<int, int>> &ranges);
int mult_solve(b200rt_ctx *c, bool reset_timer);
int mult_brightness(b200rt_ctx *c, int n_subsamples);
int mult_los_download(b200rt_ctx *c, double *const dst[4], long long stride, long long offset);
// ---- api_weights.cu
int los_weights(b200rt_ctx *c, int n_subsamples, long long *nnz);
int los_weights_nnz(b200rt_ctx *c, long long *nnz);   // B200RT_ERR_STATE unless built for the current inputs
// row_ptr[0..n_los] (+ ptr_offset), col[nnz], val[e * val_stride + p]; any may be null
int los_weights_download(b200rt_ctx *c, long long *row_ptr, long long ptr_offset, int *col, double *val, long long val_stride);
int los_weights_apply(b200rt_ctx *c, int e, int transpose, const double *x, double *y);

}  // namespace api
}  // namespace b200rt
