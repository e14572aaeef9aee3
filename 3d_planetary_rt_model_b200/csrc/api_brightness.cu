// api_brightness.cu -- line-of-sight upload, brightness (resident and pipelined host-buffer forms), download
// (one of the translation units behind the C ABI; see api_internal.hpp)
#include "api_internal.hpp"

namespace b200rt {
namespace api {
namespace {

// ------------------------------------------------------------------ brightness
// With `io` (double builds only) the lines of sight come from, and the results go to, HOST arrays.  When the set needs
// several batches (more lists than the scratch budget holds) they are pipelined -- batch b+1's nine input slices travel
// on copy_stream and batch b-1's result slices on out_stream while batch b is traversed and marched on the compute
// stream -- so that only the first upload and the last download are exposed (b200rt_brightness; with pageable host
// memory the copies degrade to staged ones, still correct).  Batches are NOT made smaller to get more overlap: a
// forced 4-way split of the 1e6-LOS bench set cost more in kernel tails (+3 ms) than the hidden copies saved (2 ms).
struct HostLos {
  int n;
  const double *const *src;   // [9]
  double *const *dst;         // [4], entries may be null
  long long out_stride;       // the caller's result arrays are [n_emissions][out_stride]; this call fills
  long long out_offset;       // [out_offset, out_offset + n) of each row (a device group hands every member a slice)
};

template <class Real>
int brightness_impl(b200rt_ctx *c, int n_subsamples, const HostLos *io = nullptr) {
  if (n_subsamples == 1 || n_subsamples < 0)
    return fail(c, B200RT_ERR_ARG, "n_subsamples must be 0 or > 1 (RT_grid.hpp:237)");
  if (io) {
    B200RT_CUDA(c, c->los_in.ensure((size_t) 9 * io->n * sizeof(Real)));
    c->n_los = io->n;
    c->los_done = false;
    c->lw.valid = false;
    if (!c->copy_stream) B200RT_CUDA(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    if (!c->out_stream) B200RT_CUDA(c, cudaStreamCreateWithFlags(&c->out_stream, cudaStreamNonBlocking));
  }
  if (c->n_los <= 0) return fail(c, B200RT_ERR_STATE, "no lines of sight uploaded");
  if (c->hg.pp)
    return fail(c, B200RT_ERR_STATE, "interp_weights not implemented in grid_plane_parallel (grid_plane_parallel.hpp:304-311)");
  for (int e = 0; e < c->n_em; e++)
    if (!c->em[e].have_S) return fail(c, B200RT_ERR_STATE, "source function not available (solve or set_sourcefn first)");
  GridView<Real> &g = gv<Real>(c);
  PhaseTimer::reset(c);
  SideStreamDrain drain(c);        // nothing stays in flight from / into the caller's arrays, error returns included
  B200RT_CUDA(c, cudaMemsetAsync(c->work_counter.p, 0, 2 * sizeof(int), c->stream));
  B200RT_CUDA(c, cudaMemsetAsync(c->step_counter.p, 0, sizeof(unsigned long long), c->stream));
  const long long n = c->n_los;
  const long long per_batch = std::min<long long>(batch_capacity(c, sizeof(Real)), n);
  ListView<Real> lv;
  if (int rc = ensure_lists<Real>(c, per_batch, &lv)) return rc;
  B200RT_CUDA(c, c->los_out.ensure((size_t) c->n_em * 4 * n * sizeof(Real)));
  B200RT_CUDA(c, c->los_order.ensure(((size_t) per_batch + 2 * (size_t) (c->hg.cap + 1)) * sizeof(int)));
  const Real *li = c->los_in.as<Real>();
  // Results for PAGEABLE caller arrays are downloaded into page-locked scratch and copied out after the stream has
  // drained: a device-to-host copy into pageable memory blocks inside the runtime until the kernels before it have
  // finished, holding a lock that stalls every other context of the process (the sweep's contexts ran their brightness
  // calls one after the other because of it).  Page-locked caller arrays (the bench's) are written directly.
  double *stage_out = nullptr;
  if (io) {
    bool pageable = false;
    for (int q = 0; q < 4 && !pageable; q++)
      if (io->dst[q]) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, io->dst[q]) != cudaSuccess) { cudaGetLastError(); pageable = true; }
        else pageable = (at.type == cudaMemoryTypeUnregistered);
      }
    if (pageable) {
      B200RT_CUDA(c, c->host_out.ensure((size_t) c->n_em * 4 * n * sizeof(double)));
      stage_out = c->host_out.as<double>();
    }
  }
  std::vector<cudaEvent_t> io_events;
  struct EventGuard {
    std::vector<cudaEvent_t> &v;
    ~EventGuard() { for (auto e : v) cudaEventDestroy(e); }
  } io_guard{io_events};
  auto io_event = [&](cudaStream_t on, cudaEvent_t *out) -> cudaError_t {   // event recorded on `on`; destroyed at return
    cudaEvent_t e;
    cudaError_t rc = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    if (rc != cudaSuccess) return rc;
    io_events.push_back(e);
    if (out) *out = e;
    return cudaEventRecord(e, on);
  };
  // the traversal reads r, z, t, cos(theta), line_z (arrays 3, 2, 4, 8, 7); x, y, line_x, line_y are only read by the
  // march, so they travel while the batch is being traversed
  cudaEvent_t uploaded_trav = nullptr, uploaded_all = nullptr;              // of the latest upload_batch
  auto upload_batch = [&](long long first) -> cudaError_t {
    const long long count = std::min(per_batch, n - first);
    static const int order_of_arrays[9] = {3, 2, 4, 8, 7, 0, 1, 5, 6};
    for (int k = 0; k < 9; k++) {
      const int a = order_of_arrays[k];
      cudaError_t rc = cudaMemcpyAsync(c->los_in.as<double>() + (size_t) a * n + first, io->src[a] + first,
                                       (size_t) count * sizeof(double), cudaMemcpyHostToDevice, c->copy_stream);
      if (rc != cudaSuccess) return rc;
      if (k == 4) {
        rc = io_event(c->copy_stream, &uploaded_trav);
        if (rc != cudaSuccess) return rc;
      }
    }
    return io_event(c->copy_stream, &uploaded_all);
  };
  EmissionView<Real> ev[MAX_EMISSIONS];
  for (int e = 0; e < c->n_em; e++) {
    ev[e] = em_view<Real>(c, e);
    Emission &E = c->em[e];
    if (E.rec_dirty) {
      B200RT_CUDA(c, launch_pack_records<Real>(ev[e], g.n_vox, E.rec_pt.as<Real>(), E.rec_avg.as<Real>(), c->stream));
      E.rec_dirty = false;
    }
  }
  int *overflow = c->work_counter.as<int>() + 1;
  for (long long first = 0; first < n; first += per_batch) {
    const long long count = std::min(per_batch, n - first);
    RayList<Real> rl;
    rl.r = li + 3 * n + first; rl.z = li + 2 * n + first; rl.t = li + 4 * n + first;
    rl.cost = li + 8 * n + first; rl.lz = li + 7 * n + first; rl.i_voxel = nullptr;
    if (io) {
      if (first == 0) B200RT_CUDA(c, upload_batch(0));
      B200RT_CUDA(c, cudaStreamWaitEvent(c->stream, uploaded_trav, 0));   // this batch's traversal slices have arrived
    }
    {
      PhaseTimer t(c, PH_TRAVERSE);
      B200RT_CUDA(c, launch_traverse_list<Real>(g, rl, count, lv, overflow, c->stream));
      t.stop(1);
    }
    if (io) B200RT_CUDA(c, cudaStreamWaitEvent(c->stream, uploaded_all, 0));
    const int *order = nullptr;
    // (a split launch that does not fit the machine at once is ordered too: its second wave then holds the short ones)
    const bool split_overflows = brightness_splits_emissions(c->n_em, count) && 2 * count > brightness_resident_groups();
    if (lv.cap <= LOS_ORDER_MAX_CAP && (count >= los_order_min() || split_overflows)) {
      PhaseTimer t(c, PH_ORDER);   // histogram, prefix, scatter: timed and counted apart from the march they feed
      int *bins = c->los_order.as<int>(), *ord = bins + 2 * (lv.cap + 1);
      B200RT_CUDA(c, launch_los_order(lv.len, count, lv.cap, bins, ord, c->stream));
      order = ord;
      t.stop(3);
    }
    {
      PhaseTimer t(c, PH_BRIGHTNESS);
      B200RT_CUDA(c, launch_brightness<Real>(g, ev, c->n_em, li, n, first, count, lv, n_subsamples,
                                             c->los_out.as<Real>(), n, c->work_counter.as<int>(),
                                             c->step_counter.as<unsigned long long>(), order, c->stream));
      t.stop(1);
    }
    if (io) {
      cudaEvent_t done;
      B200RT_CUDA(c, io_event(c->stream, &done));
      // order matters for pageable host memory, whose copies block the host: the kernels of this batch are queued
      // first, the next batch's upload runs beside them, and only then does the download wait for them
      if (first + count < n) B200RT_CUDA(c, upload_batch(first + count));
      B200RT_CUDA(c, cudaStreamWaitEvent(c->out_stream, done, 0));
      for (int e = 0; e < c->n_em; e++)
        for (int q = 0; q < 4; q++)
          if (io->dst[q])
            B200RT_CUDA(c, cudaMemcpyAsync(stage_out ? stage_out + ((size_t) e * 4 + q) * n + first
                                                     : io->dst[q] + (size_t) e * io->out_stride + io->out_offset + first,
                                           c->los_out.as<double>() + ((size_t) e * 4 + q) * n + first,
                                           (size_t) count * sizeof(double), cudaMemcpyDeviceToHost, c->out_stream));
    }
  }
  B200RT_CUDA(c, c->host_words.ensure(4 * sizeof(unsigned long long)));
  unsigned long long *substeps_p = c->host_words.as<unsigned long long>() + 1;
  B200RT_CUDA(c, cudaMemcpyAsync(substeps_p, c->step_counter.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  const int rc_overflow = check_overflow(c);
  const unsigned long long substeps = *substeps_p;
  if (io) B200RT_CUDA(c, cudaStreamSynchronize(c->out_stream));   // nothing is in flight into the caller's arrays at return
  if (rc_overflow) return rc_overflow;
  if (stage_out)
    for (int e = 0; e < c->n_em; e++)
      for (int q = 0; q < 4; q++)
        if (io->dst[q])
          std::memcpy(io->dst[q] + (size_t) e * io->out_stride + io->out_offset, stage_out + ((size_t) e * 4 + q) * n,
                      (size_t) n * sizeof(double));
  PhaseTimer::collect(c);
  c->last_substeps = (long long) substeps;
  c->los_done = true;
  return B200RT_OK;
}

template <class Real>
int los_upload_impl(b200rt_ctx *c, int n, const double *const src[9]) {
  B200RT_CUDA(c, c->los_in.ensure((size_t) 9 * n * sizeof(Real)));
  DevBuf stage;
  int rc = B200RT_OK;
  for (int a = 0; a < 9 && rc == B200RT_OK; a++)
    rc = upload_real<Real>(c, src[a], c->los_in.as<Real>() + (size_t) a * n, n, stage);
  if (rc == B200RT_OK) {
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = fail(c, B200RT_ERR_CUDA, cudaGetErrorString(e));
  }
  stage.release();
  c->n_los = n;
  c->los_done = false;
  c->lw.valid = false;
  return rc;
}

template <class Real>
int los_download_impl(b200rt_ctx *c, double *const dst[4], long long stride, long long offset) {
  const long long n = c->n_los;
  const Real *o = c->los_out.as<Real>();
  // results travel to page-locked staging in one burst and are copied out by the host: a device -> pageable copy blocks
  // inside the runtime one array at a time (and, in float, the widening happens on the way out)
  int n_arrays = 0;
  for (int q = 0; q < 4; q++) n_arrays += dst[q] != nullptr;
  if (n_arrays == 0 || n == 0) return B200RT_OK;
  B200RT_CUDA(c, c->host_out.ensure((size_t) c->n_em * n_arrays * n * sizeof(Real)));
  Real *stage = c->host_out.as<Real>();
  size_t k = 0;
  for (int e = 0; e < c->n_em; e++)
    for (int q = 0; q < 4; q++) {
      if (!dst[q]) continue;
      B200RT_CUDA(c, cudaMemcpyAsync(stage + k * n, o + ((size_t) e * 4 + q) * n, n * sizeof(Real), cudaMemcpyDeviceToHost, c->stream));
      k++;
    }
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  k = 0;
  for (int e = 0; e < c->n_em; e++)
    for (int q = 0; q < 4; q++) {
      if (!dst[q]) continue;
      double *out = dst[q] + (size_t) e * stride + offset;
      const Real *src = stage + k * n;
      if (sizeof(Real) == sizeof(double)) std::memcpy(out, src, n * sizeof(double));
      else for (long long i = 0; i < n; i++) out[i] = src[i];
      k++;
    }
  return B200RT_OK;
}


}  // namespace

int brightness_resident(b200rt_ctx *c, int n_subsamples) {
  return is64(c) ? brightness_impl<double>(c, n_subsamples) : brightness_impl<float>(c, n_subsamples);
}
int los_upload(b200rt_ctx *c, int n, const double *const src[9]) {
  return is64(c) ? los_upload_impl<double>(c, n, src) : los_upload_impl<float>(c, n, src);
}

// the slice forms need the templates above: defined here, declared in common.hpp (namespace b200rt)
int los_download_dispatch(b200rt_ctx *c, double *const dst[4], long long stride, long long offset) {
  return is64(c) ? los_download_impl<double>(c, dst, stride, offset) : los_download_impl<float>(c, dst, stride, offset);
}
int brightness_host_pipeline(b200rt_ctx *c, int n, const double *const src[9], int n_subsamples, double *const dst[4],
                             long long stride, long long offset) {
  HostLos io{n, src, dst, stride, offset};
  return brightness_impl<double>(c, n_subsamples, &io);
}

}  // namespace api

// ---- the two calls a device group hands its members with a slice of the caller's arrays (device_group.cu)
int los_download_slice(b200rt_ctx *c, double *const dst[4], long long stride, long long offset) {
  if (!c) return B200RT_ERR_ARG;
  if (!c->los_done) return fail(c, B200RT_ERR_STATE, "no brightness result to download");
  cudaSetDevice(c->device);
  if (c->mult.defined) return api::mult_los_download(c, dst, stride, offset);
  return api::los_download_dispatch(c, dst, stride, offset);
}

int brightness_slice(b200rt_ctx *c, int n, const double *const src[9], int n_subsamples, double *const dst[4],
                     long long stride, long long offset) {
  if (!c) return B200RT_ERR_ARG;
  if (api::is64(c) && !c->mult.defined && n > 0 && c->have_grid && c->n_em >= 1) {
    // double singlet model: upload, kernels and download pipelined batch by batch
    for (int a = 0; a < 9; a++) if (!src[a]) return fail(c, B200RT_ERR_ARG, "null line-of-sight array");
    cudaSetDevice(c->device);
    return api::brightness_host_pipeline(c, n, src, n_subsamples, dst, stride, offset);
  }
  int rc = b200rt_los_upload(c, n, src[0], src[1], src[2], src[3], src[4], src[5], src[6], src[7], src[8]);
  if (rc) return rc;
  rc = b200rt_brightness_resident(c, n_subsamples);
  if (rc) return rc;
  return los_download_slice(c, dst, stride, offset);
}

}  // namespace b200rt
