// los_weights.cu -- line-of-sight weighting functions: the brightness of each singlet emission as a sparse linear
// operator on its source function (sm_100a).
//
// In the brightness march (brightness.cu; reference RT_grid::brightness, RT_grid.hpp:233-299) every sub-step adds
// S_interp * gfac * T_int, with S_interp = sum_k w_k S[idx_k] the 4-corner interpolation of the source function and T_int
// a function of the emission tables and the geometry only.  So brightness_e = W_e S_e exactly, with
//   W_e[l, v] = sum over the sub-steps of l, in march order, of w_k * gfac_e * T_int_e for every corner k with idx_k == v.
// The columns of a row depend on the geometry only (the same for every emission).  Three passes per batch of lines of
// sight, on the boundary lists of traverse.cu:
//   structure (count): one warp per line of sight, the lanes take its sub-steps 32 at a time and mark the stencil
//     voxels with a nonzero weight in a per-warp bitmap of the grid (shared memory, or global scratch for large grids);
//     the popcount is the row length.  A device-wide scan of the lengths gives row_ptr.
//   structure (fill): the same marking, then the set bits in ascending order are the row's columns -- ascending and
//     unique by construction, however often the line of sight re-enters a voxel.
//   values: the brightness kernel's arithmetic unchanged (4-lane groups, both emissions in one launch), except that in
//     place of acc_B += S * gfac * T_int the lane that did a sub-step's geometry adds w_k * gfac * T_int to the slot of
//     idx_k, found by binary search in the row's sorted columns.  The sub-steps of a line of sight are applied in order
//     (one lane per sub-step, a warp barrier between them), so the values need no atomics and are the same every run.
// The whole file is compiled with FMA contraction off (Makefile): the structure and value passes evaluate the same
// stencil code, and without contraction they evaluate it to the same bits, so every voxel the value pass reads is one
// the structure pass recorded (a miss would be reported as an internal error, never dropped silently).
#include "los_march.cuh"

namespace b200rt {

namespace {

constexpr int LW_THREADS = 256;                 // structure kernels: 8 warps, one line of sight per warp at a time
constexpr int LW_WARPS = LW_THREADS / 32;
constexpr int LW_BLOCKS_PER_SM = 3;
constexpr size_t LW_SMEM_BITMAP_MAX = 64 * 1024;   // per block; larger grids keep the bitmaps in global scratch

__host__ __device__ inline size_t align16(size_t b) { return (b + 15) & ~size_t(15); }

// geometry of sub-step j of a line of sight: step length and the stencil (voxels and weights) it reads.  Restates the
// geometry half of brightness_kernel (RT_grid.hpp:262-293); without interpolation the one voxel is the current one.
template <class Real>
__device__ __forceinline__ void lw_stencil(const GeomTables<Real> &T, const Real *dl, const int *el, int j, bool interp,
                                           int nsd, int nss, Real r_nss, Real px, Real py, Real pz, Real lx, Real ly,
                                           Real lz, int (&idx)[4], Real (&w)[4], Real &s, int &cur) {
  const Real eps = MathB<Real>::eps();
  const int ib = j / nss + 1;
  const int is = j - (ib - 1) * nss + 1;
  Real d_start = dl[ib - 1];
  const Real dnext = dl[ib];
  cur = el[ib - 1];
  Real d_step = MathB<Real>::divc_(dnext - d_start, (Real) (nsd - 1), r_nss);
  d_start += Real(0.5) * eps * d_step;          // RT_grid.hpp:268-271
  d_step *= Real(1.0) - eps;
  s = d_step;
  if (!interp) {
#pragma unroll
    for (int k = 0; k < 4; k++) { idx[k] = cur; w[k] = (k == 0) ? Real(1) : Real(0); }
  } else {
    substep_interp<Real>(T, cur, px, py, pz, lx, ly, lz, d_start + is * d_step, idx, w);
  }
}

template <class Real>
struct LosPoint {
  Real px, py, pz, lx, ly, lz;   // px, py, pz already divided by the 1e9 scale
  __device__ void load(const Real *los_in, long long stride, long long los) {
    const Real scale = Real(1e9), r_scale = MathB<Real>::rcp_(scale);
    px = MathB<Real>::divc_(los_in[0 * stride + los], scale, r_scale);
    py = MathB<Real>::divc_(los_in[1 * stride + los], scale, r_scale);
    pz = MathB<Real>::divc_(los_in[2 * stride + los], scale, r_scale);
    lx = los_in[5 * stride + los]; ly = los_in[6 * stride + los]; lz = los_in[7 * stride + los];
  }
};

// ---- structure pass.  FILL = false: row lengths into row_cnt[first + t]; FILL = true: columns at row_ptr[first + t]
template <class Real, bool FILL>
__global__ void __launch_bounds__(LW_THREADS, LW_BLOCKS_PER_SM)
lw_structure_kernel(GridView<Real> g, const Real *__restrict__ los_in, long long los_stride, long long first,
                    long long count, ListView<Real> lists, int n_subsamples, int words, unsigned *gbitmap,
                    int *__restrict__ row_cnt, const long long *__restrict__ row_ptr, int *__restrict__ col) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GeomTables<Real> T;
  T.load(smem_raw, g);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned FULL = 0xffffffffu;
  unsigned *bm = gbitmap ? gbitmap + ((size_t) blockIdx.x * LW_WARPS + warp) * words
                         : reinterpret_cast<unsigned *>(smem_raw + align16(GeomTables<Real>::doubles(g.n_rb, g.n_sb) * sizeof(Real))) +
                               (size_t) warp * words;
  for (int i = lane; i < words; i += 32) bm[i] = 0;
  __syncwarp();
  const bool interp = n_subsamples != 0;
  const int nsd = interp ? n_subsamples : 2, nss = nsd - 1;
  const Real r_nss = MathB<Real>::rcp_((Real) (nsd - 1));
  for (long long t = (long long) blockIdx.x * LW_WARPS + warp; t < count; t += (long long) gridDim.x * LW_WARPS) {
    const long long los = first + t;
    const int len = lists.len[t];
    if (len <= 0) {                              // misses the grid: an empty row
      if (!FILL && lane == 0) row_cnt[los] = 0;
      continue;
    }
    const int total = (len - 1) * nss;
    const Real *dl = lists.dist + (size_t) t * lists.cap;
    const int *el = lists.ent + (size_t) t * lists.cap;
    LosPoint<Real> P;
    P.load(los_in, los_stride, los);
    int vlo = 0x7fffffff, vhi = -1;              // range of marked voxels: only those bitmap words are scanned
    for (int j = lane; j < total; j += 32) {
      int idx[4], cur;
      Real w[4], s;
      lw_stencil<Real>(T, dl, el, j, interp, nsd, nss, r_nss, P.px, P.py, P.pz, P.lx, P.ly, P.lz, idx, w, s, cur);
#pragma unroll
      for (int k = 0; k < 4; k++)
        if (w[k] != Real(0)) {
          atomicOr(&bm[idx[k] >> 5], 1u << (idx[k] & 31));
          vlo = min(vlo, idx[k]);
          vhi = max(vhi, idx[k]);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      vlo = min(vlo, __shfl_xor_sync(FULL, vlo, o));
      vhi = max(vhi, __shfl_xor_sync(FULL, vhi, o));
    }
    __syncwarp();
    const int wlo = vhi < 0 ? 0 : vlo >> 5, whi = vhi < 0 ? 0 : (vhi >> 5) + 1;
    if (!FILL) {
      int n = 0;
      for (int i = wlo + lane; i < whi; i += 32) { n += __popc(bm[i]); bm[i] = 0; }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(FULL, n, o);
      if (lane == 0) row_cnt[los] = n;
    } else {
      long long base = row_ptr[los];
      for (int i0 = wlo; i0 < whi; i0 += 32) {
        const int i = i0 + lane;
        unsigned b = (i < whi) ? bm[i] : 0u;
        const int c = __popc(b);
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int v = __shfl_up_sync(FULL, incl, o);
          if (lane >= o) incl += v;
        }
        int *out = col + base + (incl - c);
        while (b) {
          *out++ = i * 32 + (__ffs(b) - 1);
          b &= b - 1;
        }
        if (i < whi) bm[i] = 0;
        base += __shfl_sync(FULL, incl, 31);
      }
    }
    __syncwarp();
  }
}

// ---- row_ptr = exclusive scan of the row lengths (int64), in three launches: block scans, scan of the block sums, add
constexpr int SCAN_THREADS = 1024, SCAN_ITEMS = 4, SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__global__ void __launch_bounds__(SCAN_THREADS)
lw_scan_tiles_kernel(const int *__restrict__ cnt, long long n, long long *__restrict__ row_ptr, long long *__restrict__ tile_sum) {
  __shared__ long long warp_sum[32];
  const long long base = (long long) blockIdx.x * SCAN_TILE + (long long) threadIdx.x * SCAN_ITEMS;
  long long v[SCAN_ITEMS], s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++) {
    v[k] = (base + k < n) ? cnt[base + k] : 0;
    s += v[k];
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long u = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += u;
  }
  if (lane == 31) warp_sum[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    long long ws = warp_sum[lane], wi = ws;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long u = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += u;
    }
    warp_sum[lane] = wi - ws;
    if (lane == 31) tile_sum[blockIdx.x] = wi;
  }
  __syncthreads();
  long long run = warp_sum[warp] + incl - s;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++) {
    if (base + k < n) row_ptr[base + k] = run;
    run += v[k];
  }
}

__global__ void lw_scan_sums_kernel(long long *tile_sum, int n_tiles, long long *row_ptr_end) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    long long run = 0;
    for (int b = 0; b < n_tiles; b++) { const long long s = tile_sum[b]; tile_sum[b] = run; run += s; }
    *row_ptr_end = run;
  }
}

__global__ void lw_scan_add_kernel(long long *row_ptr, long long n, const long long *__restrict__ tile_sum) {
  const long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) row_ptr[i] += tile_sum[i / SCAN_TILE];
}

// ---- value pass: brightness_kernel's arithmetic with the source function replaced by the stencil's slots
template <class Real, int NEM>
__global__ void __launch_bounds__(128, (NEM == 2 && sizeof(Real) == 8) ? 3 : 4)
lw_value_kernel(GridView<Real> g, EmissionView<Real> em0, EmissionView<Real> em1, const Real *__restrict__ los_in,
                long long los_stride, long long first, long long count, ListView<Real> lists, int n_subsamples,
                const long long *__restrict__ row_ptr, const int *__restrict__ col, Real *__restrict__ val, long long nnz,
                int *queue, unsigned long long *substep_counter, const int *__restrict__ order, int *missing) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GeomTables<Real> T;
  T.load(smem_raw, g);

  const int lane = threadIdx.x & 31;
  const int sub = lane & (LPR - 1);
  const int lead = lane & ~(LPR - 1);
  const unsigned gmask = 0xFu << lead;
  const EmissionView<Real> em[2] = {em0, em1};
  const bool interp = n_subsamples != 0;
  const int nsd = interp ? n_subsamples : 2;
  const int nss = nsd - 1;
  const Real delta_lambda = Real(4.0) / (N_LAMBDA - 1);
  const Real r_nss = MathB<Real>::rcp_((Real) (nsd - 1));

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

  bool have = false, exhausted = false;
  int total = 0, j0 = 0;
  long long row_beg = 0;
  int row_len = 0;
  const Real *dl = nullptr;
  const int *el = nullptr;
  LosPoint<Real> L{};
  Real P[NEM][NLL];
  unsigned long long my_substeps = 0;
  int my_missing = 0;

  while (true) {
    while (!have && !exhausted) {
      int t = 0;
      if (sub == 0) t = atomicAdd(queue, 1);
      t = __shfl_sync(gmask, t, lead);
      if (t >= count) { exhausted = true; break; }
      if (order) t = order[t];
      const long long los = first + t;
      const int len = lists.len[t];
      if (len <= 0) continue;                      // an empty row
      total = (len - 1) * nss;
      if (sub == 0) my_substeps += (unsigned long long) total;
      dl = lists.dist + (size_t) t * lists.cap;
      el = lists.ent + (size_t) t * lists.cap;
      L.load(los_in, los_stride, los);
      row_beg = row_ptr[los];
      row_len = (int) (row_ptr[los + 1] - row_beg);
#pragma unroll
      for (int e = 0; e < NEM; e++)
#pragma unroll
        for (int m = 0; m < NLL; m++) P[e][m] = Real(1);
      j0 = 0;
      have = true;
    }
    if (__all_sync(0xffffffffu, !have)) break;

    // ---- geometry of sub-step j0+sub; the lane keeps its stencil for the adds below
    Real my_s = 0;
    Real my_in[NEM][5];
    int idx[4] = {0, 0, 0, 0};
    Real w[4] = {0, 0, 0, 0};
#pragma unroll
    for (int e = 0; e < NEM; e++)
#pragma unroll
      for (int q = 0; q < 5; q++) my_in[e][q] = 0;
    const int j = j0 + sub;
    const bool mine = have && j < total;
    if (mine) {
      int cur;
      lw_stencil<Real>(T, dl, el, j, interp, nsd, nss, r_nss, L.px, L.py, L.pz, L.lx, L.ly, L.lz, idx, w, my_s, cur);
      if (!interp) {
#pragma unroll
        for (int e = 0; e < NEM; e++) {
          const Real *r = rec_avg[e] + (size_t) cur * REC;
#pragma unroll
          for (int q = 0; q < 4; q++) my_in[e][q] = r[q];
        }
      } else {
#pragma unroll
        for (int e = 0; e < NEM; e++) interp_record<Real>(rec_pt[e], idx, w, my_in[e]);
      }
#pragma unroll
      for (int e = 0; e < NEM; e++) my_in[e][0] = LineShape<Real>::param(my_in[e][0]);
    }

    // ---- the four sub-steps in order: T_int as in brightness_kernel, then the geometry lane of the sub-step adds
    // w_k * gfac * T_int to the row slots of its stencil.  The barrier orders the adds of consecutive sub-steps.
    const unsigned FULL = 0xffffffffu;
#pragma unroll
    for (int q = 0; q < LPR; q++) {
      const Real s = shfl_real<Real>(FULL, my_s, lead + q);
      Real cT[NEM];
#pragma unroll
      for (int e = 0; e < NEM; e++) {
        const Real lsp = shfl_real<Real>(FULL, my_in[e][0], lead + q);
        const Real dts = shfl_real<Real>(FULL, my_in[e][2], lead + q);
        const Real dta = shfl_real<Real>(FULL, my_in[e][3], lead + q);
        const Real tau_species_voxel = dts * s;
        Real phi[NLL];
        LineShape<Real>::eval(lsp, sub, phi);
        Real T_int = 0;
#pragma unroll
        for (int m = 0; m < NLL; m++) {
          const Real lineshape = phi[m];
          const Real tau = (dta + dts * lineshape) * s;
          const Real tp = MathB<Real>::exp_(-tau);
          const Real c = ((double) tau < 1e-3) ? (Real(1.0) - Real(0.5) * tau) : MathB<Real>::divq_(Real(1.0) - tp, tau);
          T_int = fma(c * wgt[m], lineshape * P[e][m], T_int);
          P[e][m] *= tp;
        }
        T_int *= tau_species_voxel;
        T_int += __shfl_xor_sync(FULL, T_int, 1);
        T_int += __shfl_xor_sync(FULL, T_int, 2);
        if (T_int > tau_species_voxel) T_int = tau_species_voxel;
        cT[e] = gfac[e] * T_int;
      }
      if (sub == q && mine) {
        const int *rc = col + row_beg;
#pragma unroll
        for (int k = 0; k < 4; k++) {
          if (w[k] == Real(0)) continue;
          int lo = 0, hi = row_len;                // lower_bound of idx[k] in the row's ascending columns
          while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(rc + mid) < idx[k]) lo = mid + 1; else hi = mid;
          }
          if (lo >= row_len || __ldg(rc + lo) != idx[k]) { my_missing = 1; continue; }
#pragma unroll
          for (int e = 0; e < NEM; e++) val[(size_t) e * nnz + row_beg + lo] += w[k] * cT[e];
        }
      }
      __syncwarp();
    }
    j0 += LPR;
    if (have && j0 >= total) have = false;
  }
  if (my_missing) atomicOr(missing, 1);
  if (substep_counter) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) my_substeps += __shfl_xor_sync(0xffffffffu, my_substeps, o);
    if (lane == 0 && my_substeps) atomicAdd(substep_counter, my_substeps);
  }
}

// ---- products.  W x: one warp per row, a fixed lane-strided order and a fixed shuffle tree (the same bits every run;
// not the bits of a sequential sum)
template <class Real>
__global__ void __launch_bounds__(256)
lw_apply_kernel(const long long *__restrict__ row_ptr, const int *__restrict__ col, const Real *__restrict__ val,
                const double *__restrict__ x, long long n_rows, double *__restrict__ y) {
  const int lane = threadIdx.x & 31;
  for (long long r = ((long long) blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_rows;
       r += ((long long) gridDim.x * blockDim.x) >> 5) {
    const long long b = row_ptr[r], e = row_ptr[r + 1];
    double s = 0;
    for (long long p = b + lane; p < e; p += 32) s = fma((double) val[p], __ldg(x + col[p]), s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) y[r] = s;
  }
}

// W^T r: one warp per row scatters val * r[row] into a per-block copy of y in shared memory (atomics), which the block
// then adds into y (atomics).  Grids whose y does not fit add straight into y.  The order of the atomic adds varies from
// run to run, so the result may differ in the last bits between runs.
template <class Real>
__global__ void __launch_bounds__(256)
lw_apply_t_kernel(const long long *__restrict__ row_ptr, const int *__restrict__ col, const Real *__restrict__ val,
                  const double *__restrict__ r, long long n_rows, int n_vox, bool smem, double *__restrict__ y) {
  extern __shared__ double acc[];
  double *dst = smem ? acc : y;
  if (smem) {
    for (int v = threadIdx.x; v < n_vox; v += blockDim.x) acc[v] = 0;
    __syncthreads();
  }
  const int lane = threadIdx.x & 31;
  for (long long row = ((long long) blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < n_rows;
       row += ((long long) gridDim.x * blockDim.x) >> 5) {
    const double rv = r[row];
    if (rv == 0) continue;
    const long long b = row_ptr[row], e = row_ptr[row + 1];
    for (long long p = b + lane; p < e; p += 32) atomicAdd(dst + col[p], (double) val[p] * rv);
  }
  if (smem) {
    __syncthreads();
    for (int v = threadIdx.x; v < n_vox; v += blockDim.x)
      if (acc[v] != 0) atomicAdd(y + v, acc[v]);
  }
}

int lw_structure_blocks(long long count) {
  long long blocks = (count + LW_WARPS - 1) / LW_WARPS;
  const long long persistent = (long long) NUM_SMS * LW_BLOCKS_PER_SM;
  return (int) std::max<long long>(1, std::min(blocks, persistent));
}

} // namespace

size_t lw_bitmap_scratch_bytes(int n_vox, long long count) {
  const size_t words = ((size_t) n_vox + 31) / 32;
  if (words * 4 * LW_WARPS <= LW_SMEM_BITMAP_MAX) return 0;
  return (size_t) lw_structure_blocks(count) * LW_WARPS * words * 4;
}

template <class Real>
cudaError_t launch_lw_structure(const GridView<Real> &g, const Real *los_in, long long los_stride, long long first,
                                long long count, ListView<Real> lists, int n_subsamples, unsigned *bitmap_scratch,
                                int *row_cnt, const long long *row_ptr, int *col, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  const int words = (g.n_vox + 31) / 32;
  const bool in_smem = (size_t) words * 4 * LW_WARPS <= LW_SMEM_BITMAP_MAX;
  const size_t smem = align16(GeomTables<Real>::doubles(g.n_rb, g.n_sb) * sizeof(Real)) + (in_smem ? (size_t) words * 4 * LW_WARPS : 0);
  unsigned *gbm = in_smem ? nullptr : bitmap_scratch;
  if (!in_smem && !gbm) return cudaErrorInvalidValue;
  const int blocks = lw_structure_blocks(count);
  cudaError_t e;
  if (col) {
    e = cudaFuncSetAttribute(lw_structure_kernel<Real, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    lw_structure_kernel<Real, true><<<blocks, LW_THREADS, smem, s>>>(g, los_in, los_stride, first, count, lists, n_subsamples,
                                                                     words, gbm, row_cnt, row_ptr, col);
  } else {
    e = cudaFuncSetAttribute(lw_structure_kernel<Real, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    lw_structure_kernel<Real, false><<<blocks, LW_THREADS, smem, s>>>(g, los_in, los_stride, first, count, lists, n_subsamples,
                                                                      words, gbm, row_cnt, row_ptr, col);
  }
  return cudaGetLastError();
}

size_t lw_scan_scratch_bytes(long long n) { return (size_t) ((n + SCAN_TILE - 1) / SCAN_TILE + 1) * sizeof(long long); }

cudaError_t launch_lw_scan(const int *row_cnt, long long n, long long *row_ptr, long long *scratch, cudaStream_t s) {
  const long long tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  if (tiles > 0x7fffffffLL) return cudaErrorInvalidValue;
  if (tiles > 0) lw_scan_tiles_kernel<<<(unsigned) tiles, SCAN_THREADS, 0, s>>>(row_cnt, n, row_ptr, scratch);
  lw_scan_sums_kernel<<<1, 32, 0, s>>>(scratch, (int) tiles, row_ptr + n);
  if (n > 0) lw_scan_add_kernel<<<(unsigned) ((n + 255) / 256), 256, 0, s>>>(row_ptr, n, scratch);
  return cudaGetLastError();
}

template <class Real>
cudaError_t launch_lw_values(const GridView<Real> &g, const EmissionView<Real> *em, int n_em, const Real *los_in,
                             long long los_stride, long long first, long long count, ListView<Real> lists, int n_subsamples,
                             const long long *row_ptr, const int *col, Real *val, long long nnz, int *queue,
                             unsigned long long *substep_counter, const int *order, int *missing, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(queue, 0, sizeof(int), s);
  if (e != cudaSuccess) return e;
  const int threads = 128;
  const size_t smem = GeomTables<Real>::doubles(g.n_rb, g.n_sb) * sizeof(Real);
  long long blocks = (count * LPR + threads - 1) / threads;
  const int min_blocks = (n_em == 2 && sizeof(Real) == 8) ? 3 : 4;
  const long long persistent = (long long) NUM_SMS * min_blocks;
  if (blocks > persistent) blocks = persistent;
  if (n_em == 1) {
    e = cudaFuncSetAttribute(lw_value_kernel<Real, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    lw_value_kernel<Real, 1><<<(unsigned) blocks, threads, smem, s>>>(g, em[0], em[0], los_in, los_stride, first, count, lists,
                                                                      n_subsamples, row_ptr, col, val, nnz, queue,
                                                                      substep_counter, order, missing);
  } else {
    e = cudaFuncSetAttribute(lw_value_kernel<Real, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    lw_value_kernel<Real, 2><<<(unsigned) blocks, threads, smem, s>>>(g, em[0], em[1], los_in, los_stride, first, count, lists,
                                                                      n_subsamples, row_ptr, col, val, nnz, queue,
                                                                      substep_counter, order, missing);
  }
  return cudaGetLastError();
}

template <class Real>
cudaError_t launch_lw_apply(const long long *row_ptr, const int *col, const Real *val, long long n_rows, int n_vox,
                            int transpose, const double *x, double *y, cudaStream_t s) {
  const int threads = 256;
  const long long persistent = (long long) NUM_SMS * 8;
  long long blocks = (n_rows * 32 + threads - 1) / threads;
  blocks = std::max<long long>(1, std::min(blocks, persistent));
  if (!transpose) {
    lw_apply_kernel<Real><<<(unsigned) blocks, threads, 0, s>>>(row_ptr, col, val, x, n_rows, y);
    return cudaGetLastError();
  }
  cudaError_t e = cudaMemsetAsync(y, 0, (size_t) n_vox * sizeof(double), s);
  if (e != cudaSuccess) return e;
  const size_t smem = (size_t) n_vox * sizeof(double);
  const bool in_smem = smem <= 96 * 1024;
  if (in_smem) {
    e = cudaFuncSetAttribute(lw_apply_t_kernel<Real>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
  }
  // two blocks per SM when y sits in shared memory: every block adds its whole copy of y at the end
  if (in_smem) blocks = std::min<long long>(blocks, NUM_SMS * 2);
  lw_apply_t_kernel<Real><<<(unsigned) blocks, threads, in_smem ? smem : 0, s>>>(row_ptr, col, val, x, n_rows, n_vox, in_smem, y);
  return cudaGetLastError();
}

#define LW_INST(Real)                                                                                                      \
  template cudaError_t launch_lw_structure<Real>(const GridView<Real> &, const Real *, long long, long long, long long,    \
                                                 ListView<Real>, int, unsigned *, int *, const long long *, int *,        \
                                                 cudaStream_t);                                                           \
  template cudaError_t launch_lw_values<Real>(const GridView<Real> &, const EmissionView<Real> *, int, const Real *,        \
                                              long long, long long, long long, ListView<Real>, int, const long long *,     \
                                              const int *, Real *, long long, int *, unsigned long long *, const int *,    \
                                              int *, cudaStream_t);                                                       \
  template cudaError_t launch_lw_apply<Real>(const long long *, const int *, const Real *, long long, int, int,           \
                                             const double *, double *, cudaStream_t);
LW_INST(double)
LW_INST(float)
#undef LW_INST

} // namespace b200rt
