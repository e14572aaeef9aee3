// api_weights.cu -- line-of-sight weighting functions of the resident lines of sight: build, download, products
// (one of the translation units behind the C ABI; see api_internal.hpp; the kernels are in los_weights.cu)
#include "api_internal.hpp"

namespace b200rt {
namespace api {
namespace {

// a failed allocation of the matrix is B200RT_ERR_NOMEM (the runtime's error is not sticky: cleared here)
#define LW_ALLOC(c, call)                                                                                     \
  do {                                                                                                      \
    cudaError_t e__ = (call);                                                                               \
    if (e__ == cudaErrorMemoryAllocation) {                                                                 \
      cudaGetLastError();                                                                                   \
      return fail(c, B200RT_ERR_NOMEM, "line-of-sight weights: not enough device memory for the matrix");   \
    }                                                                                                       \
    if (e__ != cudaSuccess) return fail(c, B200RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
  } while (0)

template <class Real>
int los_weights_impl(b200rt_ctx *c, int n_subsamples, long long *nnz_out) {
  LosWeights &W = c->lw;
  W.valid = false;
  const long long n = c->n_los;
  const int n_vox = c->hg.n_vox;
  GridView<Real> &g = gv<Real>(c);
  PhaseTimer::reset(c);
  B200RT_CUDA(c, cudaMemsetAsync(c->work_counter.p, 0, 3 * sizeof(int), c->stream));
  B200RT_CUDA(c, cudaMemsetAsync(c->step_counter.p, 0, sizeof(unsigned long long), c->stream));
  const long long per_batch = std::min<long long>(batch_capacity(c, sizeof(Real)), n);
  const bool one_batch = per_batch >= n;
  ListView<Real> lv;
  if (int rc = ensure_lists<Real>(c, per_batch, &lv)) return rc;
  B200RT_CUDA(c, c->los_order.ensure(((size_t) per_batch + 2 * (size_t) (c->hg.cap + 1)) * sizeof(int)));
  LW_ALLOC(c, W.row_ptr.ensure((size_t) (n + 1) * sizeof(long long)));
  LW_ALLOC(c, W.row_cnt.ensure((size_t) n * sizeof(int)));
  LW_ALLOC(c, W.scratch.ensure(std::max(lw_scan_scratch_bytes(n), lw_bitmap_scratch_bytes(n_vox, per_batch))));
  // the brightness records of the emission tables with S = 0: the weights need no source function
  LW_ALLOC(c, W.rec.ensure((size_t) c->n_em * 2 * n_vox * 8 * sizeof(Real)));
  EmissionView<Real> ev[MAX_EMISSIONS];
  for (int e = 0; e < c->n_em; e++) {
    ev[e] = em_view<Real>(c, e);
    ev[e].sourcefn = nullptr;
    ev[e].rec_pt = W.rec.as<Real>() + (size_t) (2 * e) * n_vox * 8;
    ev[e].rec_avg = W.rec.as<Real>() + (size_t) (2 * e + 1) * n_vox * 8;
    B200RT_CUDA(c, launch_pack_records<Real>(ev[e], n_vox, const_cast<Real *>(ev[e].rec_pt), const_cast<Real *>(ev[e].rec_avg),
                                             c->stream));
  }
  const Real *li = c->los_in.as<Real>();
  int *overflow = c->work_counter.as<int>() + 1, *missing = c->work_counter.as<int>() + 2;
  auto traverse = [&](long long first, long long count) -> int {
    RayList<Real> rl;
    rl.r = li + 3 * n + first; rl.z = li + 2 * n + first; rl.t = li + 4 * n + first;
    rl.cost = li + 8 * n + first; rl.lz = li + 7 * n + first; rl.i_voxel = nullptr;
    PhaseTimer t(c, PH_TRAVERSE);
    B200RT_CUDA(c, launch_traverse_list<Real>(g, rl, count, lv, overflow, c->stream));
    t.stop(1);
    return B200RT_OK;
  };
  unsigned *bitmap = lw_bitmap_scratch_bytes(n_vox, per_batch) ? W.scratch.as<unsigned>() : nullptr;
  // ---- structure: row lengths, row_ptr
  for (long long first = 0; first < n; first += per_batch) {
    const long long count = std::min(per_batch, n - first);
    if (int rc = traverse(first, count)) return rc;
    PhaseTimer t(c, PH_LW_STRUCTURE);
    B200RT_CUDA(c, launch_lw_structure<Real>(g, li, n, first, count, lv, n_subsamples, bitmap, W.row_cnt.as<int>(),
                                             nullptr, nullptr, c->stream));
    t.stop(1);
  }
  {
    PhaseTimer t(c, PH_LW_STRUCTURE);
    B200RT_CUDA(c, launch_lw_scan(W.row_cnt.as<int>(), n, W.row_ptr.as<long long>(), W.scratch.as<long long>(), c->stream));
    t.stop(3);
  }
  B200RT_CUDA(c, c->host_words.ensure(4 * sizeof(unsigned long long)));
  long long *nnz_p = c->host_words.as<long long>() + 2;
  B200RT_CUDA(c, cudaMemcpyAsync(nnz_p, W.row_ptr.as<long long>() + n, sizeof(long long), cudaMemcpyDeviceToHost, c->stream));
  if (int rc = check_overflow(c)) return rc;      // synchronises the stream
  const long long nnz = *nnz_p;
  LW_ALLOC(c, W.col.ensure((size_t) nnz * sizeof(int)));
  LW_ALLOC(c, W.val.ensure((size_t) c->n_em * nnz * sizeof(Real)));
  B200RT_CUDA(c, cudaMemsetAsync(W.val.p, 0, (size_t) c->n_em * nnz * sizeof(Real), c->stream));
  // ---- columns and values (the lists of a single batch are still in place)
  for (long long first = 0; first < n; first += per_batch) {
    const long long count = std::min(per_batch, n - first);
    if (!one_batch)
      if (int rc = traverse(first, count)) return rc;
    {
      PhaseTimer t(c, PH_LW_STRUCTURE);
      B200RT_CUDA(c, launch_lw_structure<Real>(g, li, n, first, count, lv, n_subsamples, bitmap, nullptr,
                                               W.row_ptr.as<long long>(), W.col.as<int>(), c->stream));
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
    PhaseTimer t(c, PH_LW_VALUES);
    B200RT_CUDA(c, launch_lw_values<Real>(g, ev, c->n_em, li, n, first, count, lv, n_subsamples, W.row_ptr.as<long long>(),
                                          W.col.as<int>(), W.val.as<Real>(), nnz, c->work_counter.as<int>(),
                                          c->step_counter.as<unsigned long long>(), order, missing, c->stream));
    t.stop(1);
  }
  unsigned long long *substeps_p = c->host_words.as<unsigned long long>() + 1;
  int *missing_p = c->host_words.as<int>() + 6;
  B200RT_CUDA(c, cudaMemcpyAsync(substeps_p, c->step_counter.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  B200RT_CUDA(c, cudaMemcpyAsync(missing_p, missing, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  if (int rc = check_overflow(c)) return rc;
  if (*missing_p) return fail(c, B200RT_ERR_CUDA, "line-of-sight weights: a stencil voxel is missing from its row (internal error)");
  PhaseTimer::collect(c);
  c->last_substeps = (long long) *substeps_p;
  W.nnz = nnz;
  W.valid = true;
  if (nnz_out) *nnz_out = nnz;
  return B200RT_OK;
}

template <class Real>
int los_weights_download_impl(b200rt_ctx *c, long long *row_ptr, long long ptr_offset, int *col, double *val,
                              long long val_stride) {
  const LosWeights &W = c->lw;
  const long long n = c->n_los, nnz = W.nnz;
  if (row_ptr) {
    B200RT_CUDA(c, cudaMemcpyAsync(row_ptr, W.row_ptr.p, (size_t) (n + 1) * sizeof(long long), cudaMemcpyDeviceToHost, c->stream));
    B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
    if (ptr_offset)
      for (long long i = 0; i <= n; i++) row_ptr[i] += ptr_offset;
  }
  if (col && nnz) B200RT_CUDA(c, cudaMemcpyAsync(col, W.col.p, (size_t) nnz * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  if (val && nnz) {
    if (sizeof(Real) == sizeof(double)) {
      for (int e = 0; e < c->n_em; e++)
        B200RT_CUDA(c, cudaMemcpyAsync(val + (size_t) e * val_stride, W.val.as<Real>() + (size_t) e * nnz,
                                       (size_t) nnz * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    } else {   // widened on the host from page-locked staging
      B200RT_CUDA(c, c->host_out.ensure((size_t) c->n_em * nnz * sizeof(Real)));
      B200RT_CUDA(c, cudaMemcpyAsync(c->host_out.p, W.val.p, (size_t) c->n_em * nnz * sizeof(Real), cudaMemcpyDeviceToHost, c->stream));
      B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
      const Real *h = c->host_out.as<Real>();
      for (int e = 0; e < c->n_em; e++)
        for (long long p = 0; p < nnz; p++) val[(size_t) e * val_stride + p] = h[(size_t) e * nnz + p];
    }
  }
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  return B200RT_OK;
}

template <class Real>
int los_weights_apply_impl(b200rt_ctx *c, int e, int transpose, const double *x, double *y) {
  const LosWeights &W = c->lw;
  const long long n = c->n_los;
  const int n_vox = c->hg.n_vox;
  const long long n_in = transpose ? n : n_vox, n_out = transpose ? n_vox : n;
  B200RT_CUDA(c, c->lw.xy.ensure((size_t) (n_in + n_out) * sizeof(double)));
  double *dx = c->lw.xy.as<double>(), *dy = dx + n_in;
  PhaseTimer::reset(c);
  B200RT_CUDA(c, cudaMemcpyAsync(dx, x, (size_t) n_in * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  {
    PhaseTimer t(c, PH_LW_APPLY);
    B200RT_CUDA(c, launch_lw_apply<Real>(W.row_ptr.as<long long>(), W.col.as<int>(), W.val.as<Real>() + (size_t) e * W.nnz, n,
                                         n_vox, transpose, dx, dy, c->stream));
    t.stop(1);
  }
  B200RT_CUDA(c, cudaMemcpyAsync(y, dy, (size_t) n_out * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  PhaseTimer::collect(c);
  return B200RT_OK;
}

int lw_check_state(b200rt_ctx *c) {
  if (!c->have_grid || (c->n_em < 1 && !c->mult.defined)) return fail(c, B200RT_ERR_STATE, "grid / emissions not set");
  if (c->mult.defined) return fail(c, B200RT_ERR_STATE, "line-of-sight weights: singlet emissions only");
  if (c->hg.pp)
    return fail(c, B200RT_ERR_STATE, "interp_weights not implemented in grid_plane_parallel (grid_plane_parallel.hpp:304-311)");
  return B200RT_OK;
}

}  // namespace

int los_weights(b200rt_ctx *c, int n_subsamples, long long *nnz) {
  if (n_subsamples == 1 || n_subsamples < 0)
    return fail(c, B200RT_ERR_ARG, "n_subsamples must be 0 or > 1 (RT_grid.hpp:237)");
  if (int rc = lw_check_state(c)) return rc;
  if (c->n_los <= 0) return fail(c, B200RT_ERR_STATE, "no lines of sight uploaded");
  for (int e = 0; e < c->n_em; e++)
    if (!c->em[e].defined) return fail(c, B200RT_ERR_STATE, "emission tables not set");
  return is64(c) ? los_weights_impl<double>(c, n_subsamples, nnz) : los_weights_impl<float>(c, n_subsamples, nnz);
}

int los_weights_nnz(b200rt_ctx *c, long long *nnz) {
  if (int rc = lw_check_state(c)) return rc;
  if (!c->lw.valid) return fail(c, B200RT_ERR_STATE, "line-of-sight weights not built for the current lines of sight and tables");
  *nnz = c->lw.nnz;
  return B200RT_OK;
}

int los_weights_download(b200rt_ctx *c, long long *row_ptr, long long ptr_offset, int *col, double *val, long long val_stride) {
  long long nnz;
  if (int rc = los_weights_nnz(c, &nnz)) return rc;
  return is64(c) ? los_weights_download_impl<double>(c, row_ptr, ptr_offset, col, val, val_stride)
                 : los_weights_download_impl<float>(c, row_ptr, ptr_offset, col, val, val_stride);
}

int los_weights_apply(b200rt_ctx *c, int e, int transpose, const double *x, double *y) {
  long long nnz;
  if (int rc = los_weights_nnz(c, &nnz)) return rc;
  if (e < 0 || e >= c->n_em) return fail(c, B200RT_ERR_ARG, "bad emission index");
  return is64(c) ? los_weights_apply_impl<double>(c, e, transpose, x, y) : los_weights_apply_impl<float>(c, e, transpose, x, y);
}

}  // namespace api
}  // namespace b200rt
