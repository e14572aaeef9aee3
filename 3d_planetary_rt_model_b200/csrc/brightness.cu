// brightness.cu -- line-of-sight brightness integration (sm_100a).
//
// Restates, for the device (reference src/):
//   RT_grid::brightness(vec, los, n_subsamples)            RT_grid.hpp:233-299
//   atmo_vector::extend + atmo_point::xyz                  atmo_vec.cpp:292-306, 51-61
//   spherical_azimuthally_symmetric_grid::interp_weights   grid/grid_spherical_azimuthally_symmetric.hpp:511-612
//   emission_voxels::update_tracker_brightness_{interp,nointerp}, interp_voxel_vector
//                                                           emission/emission_voxels.hpp:58-70,199-233
//   singlet_CFR::update_tracker_start<false>, update_tracker_start_interp, update_tracker_brightness
//                                                           emission/singlet_CFR.hpp:80-260,315-348,262-276
//   los_tracker::exits_bottom                               emission/los_tracker.hpp:57-62
//
// The boundary list of each line of sight comes from traverse.cu.
//
// Mapping (the reference kernel is one LOS per thread, 32-thread blocks, tracker staged through
// shared memory; RT_gpu.cu:89-135).  Here a line of sight belongs to a GROUP of 4 lanes:
//   * the sub-steps of the LOS (segments x (n_subsamples-1)) form one flat stream that the group
//     consumes 4 at a time: lane q does the GEOMETRY of sub-step j0+q (extend, interp_weights, the
//     4-corner gathers from one interleaved 64-byte record per voxel) -- four sub-steps in parallel;
//   * then the four sub-steps are applied in order; for each, the owning lane broadcasts the
//     interpolated (q = exp(-dl^2 T), n, dtau_s, dtau_a, S, ds) with shuffles and every lane
//     integrates 5 of the 20 wavelength points (lambda index = sub + 4m), the transmission vector
//     P[5] staying in registers; the wavelength sum is two shuffles;
//   * groups pull lines of sight from a device-wide queue, so the 8 groups of a warp stay busy
//     whatever the segment counts (1..2*n_rb+n_sb) of their lines of sight are.
// In double the per-wavelength line shape exp(-lambda_i^2 T) is formed from q = exp(-dl^2 T) by
// repeated products (lambda_i = i dl => q^(i^2)): one exp per sub-step instead of 20; the products
// carry ~4e-14 relative error against a 1e-6 tolerance (float: ~1e-6 against 1e-4).
#include "los_march.cuh"

namespace b200rt {

namespace {

template <class Real>
__global__ void pack_records_kernel(const Real *__restrict__ Tr, const Real *__restrict__ dn,
                                    const Real *__restrict__ ds, const Real *__restrict__ da,
                                    const Real *__restrict__ S, int n_vox, Real *__restrict__ rec) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_vox) return;
  Real *o = rec + (size_t) v * REC;
  o[0] = Tr[v]; o[1] = dn[v]; o[2] = ds[v]; o[3] = da[v]; o[4] = S ? S[v] : Real(0); o[5] = 0; o[6] = 0; o[7] = 0;
}

#ifndef BR_MIN_BLOCKS
#define BR_MIN_BLOCKS 4
#endif
template <class Real, int NEM, bool SPLIT = false>
__global__ void __launch_bounds__(128, (NEM == 2 && sizeof(Real) == 8) ? 3 : BR_MIN_BLOCKS)
brightness_kernel(GridView<Real> g, EmissionView<Real> em0, EmissionView<Real> em1,
                  const Real *__restrict__ los_in, long long los_stride, long long first, long long count,
                  ListView<Real> lists, int n_subsamples, Real *__restrict__ out, long long n_los_total,
                  int *queue, unsigned long long *substep_counter, const int *__restrict__ order) {
  // SPLIT (NEM == 1 only): the queue holds 2 * count items, item t is line of sight t / 2 of emission t % 2
  // (em0, em1).  A small batch gives every group one line of sight whatever the order, so the launch lasts as long as
  // its longest line of sight; with the two emissions on different groups that chain is half as long.  The arithmetic
  // of an (emission, line of sight) pair is the same either way.
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GeomTables<Real> T;
  T.load(smem_raw, g);            // axes of the grid + the reciprocal tables of the double path; ends with a barrier

  const int lane = threadIdx.x & 31;
  const int sub = lane & (LPR - 1);
  const int lead = lane & ~(LPR - 1);
  const unsigned gmask = 0xFu << lead;
  const EmissionView<Real> em[2] = {em0, em1};
  const bool interp = n_subsamples != 0;
  const int nsd = interp ? n_subsamples : 2;
  const int nss = nsd - 1;                           // sub-steps per segment
  const Real eps = MathB<Real>::eps(), ceps = MathB<Real>::coneeps();
  const Real scale = Real(1e9);
  const Real delta_lambda = Real(4.0) / (N_LAMBDA - 1);
  const Real r_scale = MathB<Real>::rcp_(scale), r_nss = MathB<Real>::rcp_((Real) (nsd - 1));

  Real wgt[NLL];
#pragma unroll
  for (int m = 0; m < NLL; m++) {
    const int i = sub + LPR * m;
    wgt[m] = (i == 0 || i == N_LAMBDA - 1) ? delta_lambda : Real(2.0) * delta_lambda;
  }
  Real gfac[NEM];
  const Real *rec_pt[NEM], *rec_avg[NEM];
#pragma unroll
  for (int e = 0; e < NEM; e++) {
    gfac[e] = em[e].g_factor * em[e].branching / em[e].sigma_ref * (Real) 0.56418958354775628695 / Real(1e9);
    rec_pt[e] = em[e].rec_pt; rec_avg[e] = em[e].rec_avg;
  }
  int e_base = 0;                                    // emission of this group's line of sight when the launch is split
  const long long n_items = SPLIT ? 2 * count : count;

  // group state
  bool have = false, exhausted = false;
  long long los = 0;
  int total = 0, j0 = 0, flagbits = 0;
  const Real *dl = nullptr;
  const int *el = nullptr;
  Real px = 0, py = 0, pz = 0, lx = 0, ly = 0, lz = 0;   // px, py, pz already divided by the 1e9 scale
  Real P[NEM][NLL], acc_B[NEM], acc_tsp[NEM], acc_tab[NEM], acc_col[NEM];
  unsigned long long my_substeps = 0;

  while (true) {
    // ---- groups without work pull the next line of sight
    while (!have && !exhausted) {
      int t = 0;
      if (sub == 0) t = atomicAdd(queue, 1);
      t = __shfl_sync(gmask, t, lead);
      if (t >= n_items) { exhausted = true; break; }
      if (SPLIT) {
        e_base = t & 1;
        t >>= 1;
        const EmissionView<Real> &E = e_base ? em1 : em0;
        gfac[0] = E.g_factor * E.branching / E.sigma_ref * (Real) 0.56418958354775628695 / Real(1e9);
        rec_pt[0] = E.rec_pt;
        rec_avg[0] = E.rec_avg;
      }
      if (order) t = order[t];      // longest lines of sight first: the queue drains with short ones (launch_los_order)
      los = first + t;
      const int len = lists.len[t];
      if (len <= 0) {     // misses the grid: tracker reset values
        if (sub == 0) {
#pragma unroll
          for (int e = 0; e < NEM; e++)
#pragma unroll
            for (int q = 0; q < 4; q++) out[((size_t) (SPLIT ? e_base : e) * 4 + q) * n_los_total + los] = Real(0);
        }
        continue;
      }
      total = (len - 1) * nss;
      if (sub == 0 && (!SPLIT || e_base == 0)) my_substeps += (unsigned long long) total;
      flagbits = lists.flag[t];
      dl = lists.dist + (size_t) t * lists.cap;
      el = lists.ent + (size_t) t * lists.cap;
      px = MathB<Real>::divc_(los_in[0 * los_stride + los], scale, r_scale);
      py = MathB<Real>::divc_(los_in[1 * los_stride + los], scale, r_scale);
      pz = MathB<Real>::divc_(los_in[2 * los_stride + los], scale, r_scale);
      lx = los_in[5 * los_stride + los]; ly = los_in[6 * los_stride + los]; lz = los_in[7 * los_stride + los];
#pragma unroll
      for (int e = 0; e < NEM; e++) {
        acc_B[e] = 0; acc_tsp[e] = 0; acc_tab[e] = 0; acc_col[e] = 0;
#pragma unroll
        for (int m = 0; m < NLL; m++) P[e][m] = Real(1);
      }
      j0 = 0;
      have = true;
    }
    if (__all_sync(0xffffffffu, !have)) break;

    // ---- geometry of sub-step j0+sub (four sub-steps of the group in parallel)
    Real my_s = 0;
    Real my_in[NEM][5];
#pragma unroll
    for (int e = 0; e < NEM; e++)
#pragma unroll
      for (int q = 0; q < 5; q++) my_in[e][q] = 0;
    const int j = j0 + sub;
    if (have && j < total) {
      const int ib = j / nss + 1;
      const int is = j - (ib - 1) * nss + 1;
      Real d_start = dl[ib - 1];
      const Real dnext = dl[ib];
      const int cur = el[ib - 1];
      Real d_step = MathB<Real>::divc_(dnext - d_start, (Real) (nsd - 1), r_nss);
      d_start += Real(0.5) * eps * d_step;          // RT_grid.hpp:268-271
      d_step *= Real(1.0) - eps;
      my_s = d_step;
      if (!interp) {
#pragma unroll
        for (int e = 0; e < NEM; e++) {
          const Real *r = rec_avg[e] + (size_t) cur * REC;
#pragma unroll
          for (int q = 0; q < 5; q++) my_in[e][q] = r[q];
        }
      } else {
        int idx[4];
        Real w[4];
        const Real dist = d_start + is * d_step;
        substep_interp<Real>(T, cur, px, py, pz, lx, ly, lz, dist, idx, w);
#pragma unroll
        for (int e = 0; e < NEM; e++) interp_record<Real>(rec_pt[e], idx, w, my_in[e]);
      }
#pragma unroll
      for (int e = 0; e < NEM; e++) my_in[e][0] = LineShape<Real>::param(my_in[e][0]);
    }

    // ---- apply the four sub-steps in order.  The broadcasts and the wavelength sum are full-warp shuffles executed by
    // every lane (a group past the end of its line of sight moves garbage it never uses): with the 4-lane member masks
    // the compiler wrapped every shuffle group in MATCH / REDUX / VOTE mask checks (~5 % of the issued instructions)
    const unsigned FULL = 0xffffffffu;
#pragma unroll
    for (int q = 0; q < LPR; q++) {
      // a sub-step past the end of the line of sight has my_s == 0 and all-zero records on its lane (set above), so every
      // increment below is exactly 0: the body needs no branch, and the scheduler can overlap the tail of one sub-step
      // (shuffle reduction, clamp) with the wavelength loop of the next.  The shuffles stay unconditional (full mask).
      const Real s = shfl_real<Real>(FULL, my_s, lead + q);
#pragma unroll
      for (int e = 0; e < NEM; e++) {
        const Real lsp = shfl_real<Real>(FULL, my_in[e][0], lead + q);
        const Real dens = shfl_real<Real>(FULL, my_in[e][1], lead + q);
        const Real dts = shfl_real<Real>(FULL, my_in[e][2], lead + q);
        const Real dta = shfl_real<Real>(FULL, my_in[e][3], lead + q);
        const Real Sv = shfl_real<Real>(FULL, my_in[e][4], lead + q);
        // singlet_CFR::update_tracker_start<false> + update_tracker_brightness
        const Real tau_species_voxel = dts * s;
        acc_col[e] += dens * s;
        acc_tsp[e] += tau_species_voxel;
        acc_tab[e] += dta * s;
        Real phi[NLL];
        LineShape<Real>::eval(lsp, sub, phi);
        Real T_int = 0;
#pragma unroll
        for (int m = 0; m < NLL; m++) {
          const Real lineshape = phi[m];
          const Real tau = (dta + dts * lineshape) * s;
          const Real tp = MathB<Real>::exp_(-tau);
          const Real c = ((double) tau < 1e-3) ? (Real(1.0) - Real(0.5) * tau) : MathB<Real>::divq_(Real(1.0) - tp, tau);
          T_int = fma(c * wgt[m], lineshape * P[e][m], T_int);    // x dts * s once, after the wavelength loop
          P[e][m] *= tp;
        }
        T_int *= tau_species_voxel;
        T_int += __shfl_xor_sync(FULL, T_int, 1);
        T_int += __shfl_xor_sync(FULL, T_int, 2);
        if (T_int > tau_species_voxel) T_int = tau_species_voxel;
        acc_B[e] += Sv * gfac[e] * T_int;
      }
    }
    j0 += LPR;

    // ---- line of sight finished: write the four tracker members
    if (have && j0 >= total) {
      if (sub == 0) {
#pragma unroll
        for (int e = 0; e < NEM; e++) {
          const size_t eo = (size_t) (SPLIT ? e_base : e) * 4;
          out[(eo + 0) * n_los_total + los] = acc_B[e];
          out[(eo + 1) * n_los_total + los] = acc_tsp[e];
          out[(eo + 2) * n_los_total + los] = (flagbits & 1) ? Real(-1.0) : acc_tab[e];   // exits_bottom
          out[(eo + 3) * n_los_total + los] = acc_col[e];
        }
      }
      have = false;
    }
  }
  if (substep_counter) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) my_substeps += __shfl_xor_sync(0xffffffffu, my_substeps, o);
    if (lane == 0 && my_substeps) atomicAdd(substep_counter, my_substeps);
  }
}


// ---- longest-first order of a batch of lines of sight.  The brightness kernel is persistent (groups pull lines of
// sight from a queue) and one long line of sight takes ~0.5 ms, so in input order the last ~1.5 ms of a launch run on a
// draining machine; with the long ones first the queue ends on short ones.  Counting sort on the list length:
// (1) histogram, (2) descending exclusive prefix, (3) scatter with block-aggregated reservations.
constexpr int ORDER_THREADS = 256, ORDER_ITEMS = 16;

__global__ void __launch_bounds__(ORDER_THREADS)
los_hist_kernel(const int *__restrict__ len, long long count, int cap, int *__restrict__ hist) {
  extern __shared__ int sh_hist[];
  for (int b = threadIdx.x; b <= cap; b += ORDER_THREADS) sh_hist[b] = 0;
  __syncthreads();
  const long long base = (long long) blockIdx.x * ORDER_THREADS * ORDER_ITEMS;
  for (int k = 0; k < ORDER_ITEMS; k++) {
    const long long i = base + (long long) k * ORDER_THREADS + threadIdx.x;
    if (i < count) atomicAdd(&sh_hist[min(max(len[i], 0), cap)], 1);
  }
  __syncthreads();
  for (int b = threadIdx.x; b <= cap; b += ORDER_THREADS)
    if (sh_hist[b]) atomicAdd(&hist[b], sh_hist[b]);
}

__global__ void los_prefix_kernel(const int *__restrict__ hist, int cap, int *__restrict__ offset) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    int run = 0;
    for (int b = cap; b >= 0; b--) { offset[b] = run; run += hist[b]; }
  }
}

__global__ void __launch_bounds__(ORDER_THREADS)
los_scatter_kernel(const int *__restrict__ len, long long count, int cap, int *__restrict__ offset,
                   int *__restrict__ order) {
  extern __shared__ int sh[];
  int *sh_hist = sh, *sh_base = sh + (cap + 1);
  for (int b = threadIdx.x; b <= cap; b += ORDER_THREADS) sh_hist[b] = 0;
  __syncthreads();
  const long long base = (long long) blockIdx.x * ORDER_THREADS * ORDER_ITEMS;
  int bin[ORDER_ITEMS], rank[ORDER_ITEMS];
#pragma unroll
  for (int k = 0; k < ORDER_ITEMS; k++) {
    const long long i = base + (long long) k * ORDER_THREADS + threadIdx.x;
    bin[k] = -1;
    if (i < count) {
      bin[k] = min(max(len[i], 0), cap);
      rank[k] = atomicAdd(&sh_hist[bin[k]], 1);
    }
  }
  __syncthreads();
  for (int b = threadIdx.x; b <= cap; b += ORDER_THREADS)
    if (sh_hist[b]) sh_base[b] = atomicAdd(&offset[b], sh_hist[b]);
  __syncthreads();
#pragma unroll
  for (int k = 0; k < ORDER_ITEMS; k++)
    if (bin[k] >= 0) order[sh_base[bin[k]] + rank[k]] = (int) (base + (long long) k * ORDER_THREADS + threadIdx.x);
}

} // namespace

template <class Real>
cudaError_t launch_pack_records(const EmissionView<Real> &em, int n_vox, Real *rec_pt, Real *rec_avg, cudaStream_t s) {
  const int threads = 256, blocks = (n_vox + threads - 1) / threads;
  pack_records_kernel<Real><<<blocks, threads, 0, s>>>(em.T_ratio_pt, em.density_pt, em.dtau_species_pt,
                                                        em.dtau_absorber_pt, em.sourcefn, n_vox, rec_pt);
  pack_records_kernel<Real><<<blocks, threads, 0, s>>>(em.T_ratio, em.density, em.dtau_species, em.dtau_absorber,
                                                        em.sourcefn, n_vox, rec_avg);
  return cudaGetLastError();
}

bool brightness_splits_emissions(int n_em, long long count) {
  const char *env = getenv("B200RT_EM_SPLIT_MAX");   // read per call: the parity test switches it between two calls
  const long long split_max = env ? atoll(env) : brightness_resident_groups();
  return n_em == 2 && count <= split_max;
}
long long brightness_resident_groups() { return (long long) NUM_SMS * BR_MIN_BLOCKS * (128 / LPR); }

template <class Real>
cudaError_t launch_brightness(const GridView<Real> &g, const EmissionView<Real> *em, int n_em, const Real *los_in,
                              long long los_stride, long long first, long long count, ListView<Real> lists,
                              int n_subsamples, Real *out, long long n_los_total, int *queue,
                              unsigned long long *substep_counter, const int *order, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(queue, 0, sizeof(int), s);
  if (e != cudaSuccess) return e;
  const int threads = 128;
  const size_t smem = GeomTables<Real>::doubles(g.n_rb, g.n_sb) * sizeof(Real);
  // two emissions, few lines of sight: one emission per group (see the kernel).  The limit is the number of groups the
  // machine holds at once: beyond it groups take several lines of sight each and sharing the geometry between the
  // emissions is worth more than the shorter chain.  B200RT_EM_SPLIT_MAX overrides (0: never).
  const bool split = brightness_splits_emissions(n_em, count);
  const long long groups = split ? 2 * count : count;
  long long blocks = (groups * LPR + threads - 1) / threads;
  const long long persistent = (long long) NUM_SMS * BR_MIN_BLOCKS;   // __launch_bounds__(128, BR_MIN_BLOCKS)
  if (blocks > persistent) blocks = persistent;
  if (split) {
    e = cudaFuncSetAttribute(brightness_kernel<Real, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    brightness_kernel<Real, 1, true><<<(unsigned) blocks, threads, smem, s>>>(g, em[0], em[1], los_in, los_stride, first, count,
                                                                              lists, n_subsamples, out, n_los_total, queue, substep_counter, order);
  } else if (n_em == 1) {
    e = cudaFuncSetAttribute(brightness_kernel<Real, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    brightness_kernel<Real, 1><<<(unsigned) blocks, threads, smem, s>>>(g, em[0], em[0], los_in, los_stride, first, count,
                                                                        lists, n_subsamples, out, n_los_total, queue, substep_counter, order);
  } else {
    e = cudaFuncSetAttribute(brightness_kernel<Real, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    brightness_kernel<Real, 2><<<(unsigned) blocks, threads, smem, s>>>(g, em[0], em[1], los_in, los_stride, first, count,
                                                                        lists, n_subsamples, out, n_los_total, queue, substep_counter, order);
  }
  return cudaGetLastError();
}
template cudaError_t launch_brightness<double>(const GridView<double> &, const EmissionView<double> *, int,
                                               const double *, long long, long long, long long, ListView<double>, int,
                                               double *, long long, int *, unsigned long long *, const int *, cudaStream_t);
template cudaError_t launch_brightness<float>(const GridView<float> &, const EmissionView<float> *, int, const float *,
                                              long long, long long, long long, ListView<float>, int, float *,
                                              long long, int *, unsigned long long *, const int *, cudaStream_t);
cudaError_t launch_los_order(const int *len, long long count, int cap, int *bins, int *order, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  if (cap > LOS_ORDER_MAX_CAP || count > 0x7fffffffLL) return cudaErrorInvalidValue;
  int *hist = bins, *offset = bins + (cap + 1);
  cudaError_t e = cudaMemsetAsync(hist, 0, (size_t) (cap + 1) * sizeof(int), s);
  if (e != cudaSuccess) return e;
  const long long per_block = (long long) ORDER_THREADS * ORDER_ITEMS;
  const unsigned blocks = (unsigned) ((count + per_block - 1) / per_block);
  los_hist_kernel<<<blocks, ORDER_THREADS, (size_t) (cap + 1) * sizeof(int), s>>>(len, count, cap, hist);
  los_prefix_kernel<<<1, 32, 0, s>>>(hist, cap, offset);
  e = cudaFuncSetAttribute(los_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) (2 * (cap + 1) * sizeof(int)));
  if (e != cudaSuccess) return e;
  los_scatter_kernel<<<blocks, ORDER_THREADS, (size_t) 2 * (cap + 1) * sizeof(int), s>>>(len, count, cap, offset, order);
  return cudaGetLastError();
}

template cudaError_t launch_pack_records<double>(const EmissionView<double> &, int, double *, double *, cudaStream_t);
template cudaError_t launch_pack_records<float>(const EmissionView<float> &, int, float *, float *, cudaStream_t);

} // namespace b200rt
