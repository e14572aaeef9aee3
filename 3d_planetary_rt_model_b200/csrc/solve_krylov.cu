// solve_krylov.cu -- (I - w K) S = S0 with the rows of K left on the GPUs that built them (sm_100a).
//
// The reference solves the dense system on one device (emission_voxels::solve_gpu, cuSOLVER getrf/getrs,
// emission_voxels.hpp:293-340); solve.cu is that path here (block LU, DMMA).  With the influence rows built on N GPUs the
// LU is what the other N-1 wait for, and its input has to be gathered first.  This file is the N-GPU form of the solve:
// K is the kernel of a second-kind integral equation, its spectrum clusters at 0, so GMRES on I - wK converges in a
// number of steps that does not grow with the grid (measured with the CPU oracle, tools/dev/krylov_probe.py: 66 steps to
// 1e-12, 78 to 1e-14 on both the 40x20 and the 100x60 grid; rho(wK) = 0.97, so the plain Neumann series needs ~900).
// One step = one product with K: every rank multiplies ITS rows (n_vox^2 * 8 / N bytes from HBM, ~6 us on eight B200s),
// writes its piece of the result straight into every rank's exchange block (peer stores over NVLink: plain peer access
// inside a process, CUDA IPC between processes) and posts a round counter there; every rank then orthogonalises the
// assembled vector redundantly with the same kernels in the same order, so the Krylov bases -- and the step at which the
// iteration stops -- are bit-identical on all ranks and nothing else is ever exchanged.  No row gather, no broadcast of
// S, no host barrier: the only synchronisation is a kernel of rank r waiting for the round counters of its peers.
//
// Three parts below.  (1) The algorithm as separate launches, four per step -- the first form built, kept as the fallback
// when a cooperative launch does not fit (B200RT_KRYLOV_FUSED=0 selects it; it iterates on A itself):
//     kry_post<1>  x = w / |w| -> V[j];  (x - w K x)[own rows] -> every block;  post round
//     kry_orth<0>  wait for the round;  w = assembled vector;  partial V^T w per slice
//     kry_orth<1>  h1 = sum of partials;  w -= V h1;  partial V^T w          (classical Gram-Schmidt, twice)
//     kry_orth<2>  h2;  w -= V h2;  |w|^2 partials;  last CTA: Hessenberg column, Givens, residual, stop?
// (2) The right preconditioner's set-up (kry_pre_*): diagonal blocks of A over the SZA columns, inverted on every rank, and
// the own rows of A M^-1.  (3) kry_loop: the whole iteration as ONE cooperative launch per rank -- the default.
// All sums run in a fixed order (no floating-point atomics): deterministic, and identical on every rank.
// The round counters are monotonic over the life of a block and every rank runs the same rounds, so they never need
// resetting; the vector slots alternate with the round (a rank can be at most one round ahead of a peer that still reads).
#include <cstddef>
#include <cstdio>
#include <mutex>
#include "api_internal.hpp"

namespace b200rt {

namespace {

constexpr int KRY_MAX_IT = 160;                      // Arnoldi steps (basis vectors) before giving up
constexpr int KRY_SLICE = 96;                        // elements of the vector one CTA of the orthogonalisation owns
constexpr int KRY_THREADS = 256;
constexpr int KRY_WARPS = KRY_THREADS / 32;
constexpr int KRY_VPT = 8;                            // basis vectors a warp has in flight per trip (L2 latency)
constexpr int KRY_MAX_N = B200RT_KRYLOV_MAX_N;       // 24576 unknowns: the exchange block has a fixed layout
constexpr int KRY_MAX_WORLD = B200RT_KRYLOV_MAX_WORLD;
constexpr int KRY_MAX_B = (KRY_MAX_N + KRY_SLICE - 1) / KRY_SLICE;

constexpr int KRY_MAX_NR = B200RT_KRYLOV_MAX_NR;     // unknowns of one diagonal block of the preconditioner (128)
struct KryExchange {                                 // one per rank, written by every rank
  unsigned long long flag[KRY_MAX_WORLD][16];        // flag[q][0]: rounds rank q has completed into THIS block (own 128-byte line)
  double w[2][KRY_MAX_N];
  double pre[(size_t) KRY_MAX_N * KRY_MAX_NR];       // pre[e][i']: A[e][unknown i' of the block of e], the diagonal blocks
                                                     // of the preconditioner, every row written by the rank that built it
};
static_assert(sizeof(KryExchange) == B200RT_KRYLOV_BLOCK_BYTES, "include/b200rt.h states the size of the exchange block");

struct KryPeers {
  KryExchange *p[KRY_MAX_WORLD];
  int rank, world;
};

struct KryState {
  unsigned long long round;          // rounds this rank has posted (monotonic; equal on all ranks between solves)
  int iter, done, error, converged;
  unsigned int post_tickets, orth_tickets, row_queue;
  int max_it;
  double beta, inv_norm, res, true_res, tol;
  // the one-launch form (kry_loop): barrier among the CTAs that orthogonalise, and the step sequence CTA 0 publishes
  unsigned int orth_bar, step_seq;
  unsigned long long t_phase[10];    // CTA 0's clock over the Arnoldi steps [ns]: product, wait for peers, orthogonalisation,
                                     // closing; [4..9]: the orthogonalisation's three passes and the barrier after each
};

struct KryWork {                     // device pointers into one allocation
  KryState *st;
  double *V;                         // [KRY_MAX_IT + 1][ns]
  double *wloc, *bvec, *xsol;        // [ns]
  double *part1, *part2;             // [KRY_MAX_IT + 1][KRY_MAX_B]
  double *npart;                     // [KRY_MAX_B]
  double *R;                         // [KRY_MAX_IT + 1][KRY_MAX_IT], upper triangular after the rotations
  double *cs, *sn, *g, *y;           // [KRY_MAX_IT + 1]
  int ns;
  // right preconditioner M = diagonal blocks of A.  Unknown e = voxel * nu + state, voxel = i_r * n_col + i_col; the
  // COLUMN ORDER p = i_col * cl + i_r * nu + state (cl = n_r * nu) lists every SZA column's unknowns radially outwards, and
  // each column is cut into n_runs runs of `run` unknowns (whole voxels; the last run is shorter where run does not divide cl): block
  // b = i_col * n_runs + k covers positions [i_col * cl + k * run, + min(run, cl - k * run)).  One state and n_r <= 128:
  // one block per SZA column.
  double *Minv;                      // [n_col * n_runs][run * run] the inverted blocks (every rank inverts all of them, identically)
  double *Bp;                        // [own rows][n] rows of A M^-1, columns in the column order
  double *usol;                      // [ns] V y before M^-1 is applied
  double *wperm;                     // [ns] the current vector in the column order of Bp (what the product reads)
  int run, n_col, nu, cl, n_runs;    // run = 0: no preconditioner
};

__device__ __forceinline__ int pc_perm(const KryWork &wk, int e) {    // unknown -> position in the column order
  const int v = e / wk.nu, s = e - v * wk.nu, ir = v / wk.n_col, ic = v - ir * wk.n_col;
  return ic * wk.cl + ir * wk.nu + s;
}
__device__ __forceinline__ int pc_elem(const KryWork &wk, int p) {    // position in the column order -> unknown
  const int ic = p / wk.cl, q = p - ic * wk.cl, ir = q / wk.nu, s = q - ir * wk.nu;
  return (ir * wk.n_col + ic) * wk.nu + s;
}
__device__ __forceinline__ int pc_block_of(const KryWork &wk, int p) {
  const int ic = p / wk.cl;
  return ic * wk.n_runs + (p - ic * wk.cl) / wk.run;
}
__device__ __forceinline__ void pc_block(const KryWork &wk, int b, int *p0, int *len) {   // first position, unknowns
  const int ic = b / wk.n_runs, k = b - ic * wk.n_runs;
  *p0 = ic * wk.cl + k * wk.run;
  *len = min(wk.run, wk.cl - k * wk.run);
}

__device__ __forceinline__ unsigned long long ld_flag(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_flag_relaxed(unsigned long long *p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// the round flag: a system-scope release by the posting thread (one thread per peer, all at once), so that everything this
// CTA has observed -- every CTA's pieces, already fenced system-wide by their authors -- is ordered before the flag for
// the peer that acquires it
__device__ __forceinline__ void st_flag_release(unsigned long long *p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ double ld_remote(const double *p) {       // written by a peer: never through L1
  double v;
  asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_remote(double *p, double v) {
  asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// MODE 0: the right-hand side (S0 of the own rows, so that every rank starts from the same bits)
// MODE 1: an Arnoldi step: x = wloc * inv_norm is basis vector `iter`;  (x - w K x)[own rows]
// MODE 2: the residual check: (x - w K x)[own rows] for x = the solution
// A CTA takes rows from a queue, one at a time: the row streams from HBM once (evict-first loads, 8 in flight per thread),
// x (47 kB) is read through L1 where every CTA of the SM finds it; the scale 1/|w| is applied to the sum, not to the
// 5841 operands.  The grid is as many CTAs as the machine holds (or as there are rows): measured, a warp per row left a
// quarter-filled second wave running at the latency-bound rate (94 us per product), a CTA per row paid two system-wide
// fences and a ticket per row (79 us for the 5841 rows of one GPU even without the product).
template <int MODE>
__global__ void __launch_bounds__(KRY_THREADS)
kry_post(const double *__restrict__ K, int n, const int *__restrict__ rows, int n_rows, double branching,
         const double *__restrict__ S0, KryWork wk, KryPeers pe) {
  KryState *st = wk.st;
  if (MODE == 1 && st->done) return;
  __shared__ double red[KRY_WARPS];
  __shared__ int sh_row;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned long long round = st->round;      // (the last CTA advances it after every CTA has taken its ticket)
  const int slot = (int) (round & 1);
  const double *src = MODE == 1 ? wk.wloc : wk.xsol;
  const double scale = MODE == 1 ? st->inv_norm : 1.0;
  if (MODE == 1) {                                 // the grid stores the new basis vector, a chunk per CTA
    const int chunk = (n + gridDim.x - 1) / gridDim.x;
    const int lo = blockIdx.x * chunk, hi = min(n, lo + chunk);
    double *Vj = wk.V + (size_t) st->iter * wk.ns;
    for (int i = lo + tid; i < hi; i += KRY_THREADS) Vj[i] = src[i] * scale;
  }
  for (;;) {
    if (tid == 0) sh_row = (int) atomicAdd(&st->row_queue, 1u);
    __syncthreads();
    const int slot_row = sh_row;
    if (slot_row >= n_rows) break;
    const int i = rows[slot_row];
    double val = 0;
    if (MODE == 0) {
      val = S0[i];
    } else {
      const double *Kr = K + (size_t) i * n;
      double acc[8];
#pragma unroll
      for (int u = 0; u < 8; u++) acc[u] = 0;
      int col = tid;
      for (; col + 7 * KRY_THREADS < n; col += 8 * KRY_THREADS) {
        double k8[8];
#pragma unroll
        for (int u = 0; u < 8; u++) k8[u] = __ldcs(Kr + col + KRY_THREADS * u);
#pragma unroll
        for (int u = 0; u < 8; u++) acc[u] = fma(k8[u], __ldg(src + col + KRY_THREADS * u), acc[u]);
      }
#pragma unroll
      for (int u = 0; u < 8; u++) {                  // the last, partial trip
        const int cc = col + KRY_THREADS * u;
        if (cc < n) acc[u] = fma(__ldcs(Kr + cc), __ldg(src + cc), acc[u]);
      }
      double s = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) red[warp] = s;
      __syncthreads();
      if (tid < 32) {
        double t = 0;
#pragma unroll
        for (int k = 0; k < KRY_WARPS; k++) t += red[k];
        val = scale * (__ldg(src + i) - branching * t);
      }
    }
    if (tid < pe.world) st_remote(&pe.p[tid]->w[slot][i], val);
    __syncthreads();                               // red[] and sh_row are reused by the next row
  }
  if (tid < pe.world) __threadfence_system();      // this CTA's pieces are in the peers' memory before its ticket
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    const unsigned int t = atomicAdd(&st->post_tickets, 1u);
    sh_row = (t == gridDim.x - 1);
    if (sh_row) {                                  // every CTA's pieces are out
      __threadfence();
      st->post_tickets = 0;
      st->row_queue = 0;
      st->round = round + 1;
    }
  }
  __syncthreads();
  if (sh_row && tid < pe.world) {                  // post the round on every rank, one thread per peer
    if (MODE == 0) st_flag_relaxed(&pe.p[tid]->flag[pe.rank][1], (unsigned long long) n_rows);   // row census, read after the round
    st_flag_release(&pe.p[tid]->flag[pe.rank][0], round + 1);
  }
}

// ---- pieces of the orthogonalisation; a CTA owns elements [lo, lo + len) of the vector, ws[] is its copy
// partial dot products of the slice with basis vectors 0 .. nv-1 -> part[v][cta]
__device__ __forceinline__ void slice_dots(const double *ws, const KryWork &wk, int lo, int len, int nv, double *part) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double wr[KRY_SLICE / 32];
#pragma unroll
  for (int u = 0; u < KRY_SLICE / 32; u++) wr[u] = (lane + 32 * u < len) ? ws[lane + 32 * u] : 0.0;
  for (int v0 = warp; v0 < nv; v0 += KRY_VPT * KRY_WARPS) {      // KRY_VPT basis vectors per trip: their loads overlap (L2 latency)
    double vv[KRY_VPT][KRY_SLICE / 32];
#pragma unroll
    for (int k = 0; k < KRY_VPT; k++) {
      const int v = v0 + k * KRY_WARPS;
      const double *Vv = wk.V + (size_t) min(v, nv - 1) * wk.ns + lo;
#pragma unroll
      for (int u = 0; u < KRY_SLICE / 32; u++) vv[k][u] = (lane + 32 * u < len) ? Vv[lane + 32 * u] : 0.0;
    }
    double s[KRY_VPT];
#pragma unroll
    for (int k = 0; k < KRY_VPT; k++) {
      s[k] = 0;
#pragma unroll
      for (int u = 0; u < KRY_SLICE / 32; u++) s[k] = fma(vv[k][u], wr[u], s[k]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int k = 0; k < KRY_VPT; k++) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
#pragma unroll
    for (int k = 0; k < KRY_VPT; k++)
      if (lane == 0 && v0 + k * KRY_WARPS < nv) part[(size_t) (v0 + k * KRY_WARPS) * KRY_MAX_B + blockIdx.x] = s[k];
  }
}
// sum over the CTAs of p[0 .. n_cta): a warp, lane c taking p[c], p[c + 32], ... and a fixed shuffle tree (the same order
// on every rank); valid on every lane
__device__ __forceinline__ double warp_sum_partials(const double *p, int n_cta) {
  const int lane = threadIdx.x & 31;
  double s = 0;
  for (int c = lane; c < n_cta; c += 32) s += p[c];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  return s;
}
// h[v] = sum over the CTAs of part[v][.]
__device__ __forceinline__ void slice_reduce(const double *part, int nv, int n_cta, double *h) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int v0 = warp; v0 < nv; v0 += KRY_VPT * KRY_WARPS) {
    double s[KRY_VPT];
#pragma unroll
    for (int k = 0; k < KRY_VPT; k++) {
      const double *p = part + (size_t) min(v0 + k * KRY_WARPS, nv - 1) * KRY_MAX_B;
      s[k] = 0;
      for (int c = lane; c < n_cta; c += 32) s[k] += p[c];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int k = 0; k < KRY_VPT; k++) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
#pragma unroll
    for (int k = 0; k < KRY_VPT; k++)
      if (lane == 0 && v0 + k * KRY_WARPS < nv) h[v0 + k * KRY_WARPS] = s[k];
  }
}
// ws -= sum_v h[v] V[v][slice]: warp k sums the vectors v = k mod 8, then the eight partial sums are added in order
__device__ __forceinline__ void slice_update(double *ws, const KryWork &wk, int lo, int len, int nv, const double *h,
                                             double (*red)[KRY_SLICE], double sign) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double acc[KRY_SLICE / 32];
#pragma unroll
  for (int u = 0; u < KRY_SLICE / 32; u++) acc[u] = 0;
  for (int v0 = warp; v0 < nv; v0 += KRY_VPT * KRY_WARPS) {
    double vv[KRY_VPT][KRY_SLICE / 32], hv[KRY_VPT];
#pragma unroll
    for (int k = 0; k < KRY_VPT; k++) {
      const int v = v0 + k * KRY_WARPS;
      const double *Vv = wk.V + (size_t) min(v, nv - 1) * wk.ns + lo;
      hv[k] = v < nv ? h[v] : 0.0;
#pragma unroll
      for (int u = 0; u < KRY_SLICE / 32; u++) vv[k][u] = (lane + 32 * u < len) ? Vv[lane + 32 * u] : 0.0;
    }
#pragma unroll
    for (int k = 0; k < KRY_VPT; k++)
#pragma unroll
      for (int u = 0; u < KRY_SLICE / 32; u++) acc[u] = fma(hv[k], vv[k][u], acc[u]);
  }
#pragma unroll
  for (int u = 0; u < KRY_SLICE / 32; u++) red[warp][lane + 32 * u] = acc[u];
  __syncthreads();
  if ((int) threadIdx.x < len) {
    double s = 0;
#pragma unroll
    for (int k = 0; k < KRY_WARPS; k++) s += red[k][threadIdx.x];
    ws[threadIdx.x] += sign * s;
  }
  __syncthreads();
}
// sum over the slice of f, in a fixed order; valid on thread 0
__device__ __forceinline__ double slice_sum(double f, double *scratch) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) f += __shfl_xor_sync(0xffffffffu, f, o);
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = f;
  __syncthreads();
  double s = 0;
  if (threadIdx.x == 0)
    for (int k = 0; k < KRY_WARPS; k++) s += scratch[k];
  __syncthreads();
  return s;
}
// thread 0 waits until every rank has posted `round` into this rank's block; false (and st->error) after 20 s
__device__ __forceinline__ bool wait_round(KryState *st, const KryPeers &pe, unsigned long long round, int *sh_ok) {
  if (threadIdx.x == 0) {
    const KryExchange *mine = pe.p[pe.rank];
    const unsigned long long t0 = global_ns();
    int ok = 1;
    for (int q = 0; q < pe.world && ok; q++) {
      unsigned int spins = 0;
      while (ld_flag(&mine->flag[q][0]) < round) {
        __nanosleep(64);
        if ((++spins & 1023u) == 0 && global_ns() - t0 > 20000000000ull) { ok = 0; break; }
      }
    }
    if (!ok) { st->error = 1; st->done = 1; }
    *sh_ok = ok;
  }
  __syncthreads();
  return *sh_ok != 0;
}
// true on the CTA that finishes last (all threads)
__device__ __forceinline__ bool last_cta(KryState *st, int *sh_last) {
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int t = atomicAdd(&st->orth_tickets, 1u);
    *sh_last = (t == gridDim.x - 1);
    if (*sh_last) { st->orth_tickets = 0; __threadfence(); }
  }
  __syncthreads();
  return *sh_last != 0;
}

// after kry_post<0>: b = the assembled right-hand side, beta = |b|, first residual vector = b
__global__ void __launch_bounds__(KRY_THREADS)
kry_begin(int n, KryWork wk, KryPeers pe, double tol, int max_it) {
  __shared__ double scratch[KRY_WARPS];
  __shared__ int sh_flag;
  KryState *st = wk.st;
  const int tid = threadIdx.x;
  const unsigned long long round = st->round;
  if (!wait_round(st, pe, round, &sh_flag)) return;
  const int slot = (int) ((round - 1) & 1);
  const int lo = blockIdx.x * KRY_SLICE, len = min(KRY_SLICE, n - lo);
  double b = 0;
  if (tid < len) {
    b = ld_remote(&pe.p[pe.rank]->w[slot][lo + tid]);
    wk.bvec[lo + tid] = b;
    wk.wloc[lo + tid] = b;
  }
  const double s = slice_sum(b * b, scratch);
  if (tid == 0) wk.npart[blockIdx.x] = s;
  const bool last = last_cta(st, &sh_flag);
  if (last && tid < 32) {
    const double t = warp_sum_partials(wk.npart, gridDim.x);
    if (tid == 0) scratch[0] = t;
  }
  __syncthreads();
  if (last && tid == 0) {
    const double beta = sqrt(scratch[0]);
    st->beta = beta;
    st->inv_norm = beta > 0 ? 1.0 / beta : 0.0;
    wk.g[0] = beta;
    st->iter = 0;
    st->res = 1.0;
    st->true_res = -1.0;
    st->tol = tol;
    st->max_it = max_it;
    st->converged = beta > 0 ? 0 : 1;       // S0 = 0: S = 0
    st->done = beta > 0 ? 0 : 1;
    unsigned long long census = 0;           // the ranks' rows must add up to the grid
    for (int q = 0; q < pe.world; q++) census += ld_flag(&pe.p[pe.rank]->flag[q][1]);
    if (census != (unsigned long long) n) { st->error = 2; st->done = 1; }
  }
}

// PASS 0: wait, take the assembled vector, first partial V^T w.   PASS 1: w -= V h1, second partial V^T w.
// PASS 2: w -= V h2, |w|^2; the last CTA closes the step (Hessenberg column, Givens rotation, residual estimate).
template <int PASS>
__global__ void __launch_bounds__(KRY_THREADS)
kry_orth(int n, KryWork wk, KryPeers pe) {
  __shared__ double ws[KRY_SLICE];
  __shared__ double red[KRY_WARPS][KRY_SLICE];
  __shared__ double h[KRY_MAX_IT + 2];
  __shared__ double scratch[KRY_WARPS];
  __shared__ int sh_flag;
  KryState *st = wk.st;
  if (st->done) return;
  const int tid = threadIdx.x;
  const int lo = blockIdx.x * KRY_SLICE, len = min(KRY_SLICE, n - lo);
  const int j = st->iter, nv = j + 1;          // basis vectors 0 .. j exist
  if (PASS == 0) {
    const unsigned long long round = st->round;
    if (!wait_round(st, pe, round, &sh_flag)) return;
    const int slot = (int) ((round - 1) & 1);
    if (tid < len) ws[tid] = ld_remote(&pe.p[pe.rank]->w[slot][lo + tid]);
    __syncthreads();
    slice_dots(ws, wk, lo, len, nv, wk.part1);
    if (tid < len) wk.wloc[lo + tid] = ws[tid];
    return;
  }
  if (tid < len) ws[tid] = wk.wloc[lo + tid];
  slice_reduce(PASS == 1 ? wk.part1 : wk.part2, nv, gridDim.x, h);
  __syncthreads();
  slice_update(ws, wk, lo, len, nv, h, red, -1.0);
  if (tid < len) wk.wloc[lo + tid] = ws[tid];
  if (PASS == 1) {
    slice_dots(ws, wk, lo, len, nv, wk.part2);
    return;
  }
  const double w2 = slice_sum(tid < len ? ws[tid] * ws[tid] : 0.0, scratch);
  if (tid == 0) wk.npart[blockIdx.x] = w2;
  if (!last_cta(st, &sh_flag)) return;
  // ---- close step j: column j of the Hessenberg matrix is h1 + h2 (both Gram-Schmidt passes) and |w|
  {
    const int lane = tid & 31, warp = tid >> 5;
    double *h1 = &red[4][0];                         // (red is free here: 8 x 96 doubles)
    slice_reduce(wk.part1, nv, gridDim.x, h1);       // h still holds h2, the sums of part2
    __syncthreads();
    for (int v = tid; v < nv; v += KRY_THREADS) h[v] = h1[v] + h[v];
    if (warp == 0) {
      const double t = warp_sum_partials(wk.npart, gridDim.x);
      if (lane == 0) scratch[0] = t;
    }
    double *rot = &red[0][0];                       // the rotations so far, staged for the serial sweep below
    for (int i = tid; i < j; i += KRY_THREADS) { rot[2 * i] = wk.cs[i]; rot[2 * i + 1] = wk.sn[i]; }
  }
  __syncthreads();
  if (tid == 0) {
    const double *rot = &red[0][0];
    const double hn = sqrt(scratch[0]);
    double hi = h[0];                               // the element the next rotation mixes with h[i + 1]
    for (int i = 0; i < j; i++) {
      const double c_ = rot[2 * i], s_ = rot[2 * i + 1], up = h[i + 1];
      h[i] = c_ * hi + s_ * up;
      hi = -s_ * hi + c_ * up;
    }
    const double d = hypot(hi, hn);
    const double c_ = d > 0 ? hi / d : 1.0, s_ = d > 0 ? hn / d : 0.0;
    h[j] = d;
    wk.cs[j] = c_; wk.sn[j] = s_;
    const double gj = wk.g[j];
    wk.g[j + 1] = -s_ * gj;
    wk.g[j] = c_ * gj;
    const double res = fabs(wk.g[j + 1]) / st->beta;
    st->res = res;
    st->iter = j + 1;
    st->inv_norm = hn > 0 ? 1.0 / hn : 0.0;
    const bool conv = res <= st->tol || hn == 0.0;
    st->converged = conv ? 1 : 0;
    st->done = (conv || j + 1 >= st->max_it) ? 1 : 0;
  }
  __syncthreads();
  for (int i = tid; i <= j; i += KRY_THREADS) wk.R[(size_t) i * KRY_MAX_IT + j] = h[i];
}

// y = R^-1 g (k = iter unknowns), one warp
__global__ void kry_backsolve(KryWork wk) {
  const int k = wk.st->iter, lane = threadIdx.x;
  for (int i = k - 1; i >= 0; i--) {
    double s = 0;
    for (int l = i + 1 + lane; l < k; l += 32) s = fma(wk.R[(size_t) i * KRY_MAX_IT + l], wk.y[l], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) wk.y[i] = (wk.g[i] - s) / wk.R[(size_t) i * KRY_MAX_IT + i];
    __syncwarp();
  }
}
// S = V y
__global__ void __launch_bounds__(KRY_THREADS)
kry_solution(int n, KryWork wk, double *__restrict__ S) {
  __shared__ double ws[KRY_SLICE];
  __shared__ double red[KRY_WARPS][KRY_SLICE];
  __shared__ double h[KRY_MAX_IT + 2];
  const int tid = threadIdx.x;
  const int lo = blockIdx.x * KRY_SLICE, len = min(KRY_SLICE, n - lo);
  const int k = wk.st->iter;
  for (int v = tid; v < k; v += KRY_THREADS) h[v] = wk.y[v];
  if (tid < KRY_SLICE) ws[tid] = 0;
  __syncthreads();
  slice_update(ws, wk, lo, len, k, h, red, 1.0);
  if (tid < len) { wk.xsol[lo + tid] = ws[tid]; S[lo + tid] = ws[tid]; }
}
// after kry_post<2>: |b - (I - wK) S| / |b|
__global__ void __launch_bounds__(KRY_THREADS)
kry_residual(int n, KryWork wk, KryPeers pe) {
  __shared__ double scratch[KRY_WARPS];
  __shared__ int sh_flag;
  KryState *st = wk.st;
  const int tid = threadIdx.x;
  const unsigned long long round = st->round;
  if (st->error) return;
  if (!wait_round(st, pe, round, &sh_flag)) return;
  const int slot = (int) ((round - 1) & 1);
  const int lo = blockIdx.x * KRY_SLICE, len = min(KRY_SLICE, n - lo);
  double r = 0;
  if (tid < len) r = wk.bvec[lo + tid] - ld_remote(&pe.p[pe.rank]->w[slot][lo + tid]);
  const double s = slice_sum(r * r, scratch);
  if (tid == 0) wk.npart[blockIdx.x] = s;
  if (last_cta(st, &sh_flag) && tid < 32) {
    const double t = warp_sum_partials(wk.npart, gridDim.x);
    if (tid == 0) st->true_res = st->beta > 0 ? sqrt(t) / st->beta : 0.0;
  }
}

// =====================================================================================================================
// Right preconditioner: M = the diagonal blocks of A = I - wK over the SZA columns of the grid (all radial voxels of one
// SZA index: the strongest coupling in this atmosphere is vertical).  GMRES on A M^-1 u = S0, S = M^-1 u: 39 steps
// instead of 71 on the 100x60 grid, 24 instead of 69 on the 40x20 grid (tools/dev/krylov_probe.py); residuals are those
// of the original system.  Three launches before the iteration:
//   kry_pre_post    every rank writes the block entries of ITS rows into every rank's exchange block (one more round);
//   kry_pre_invert  every rank inverts all n_col blocks (nr x nr, Gauss-Jordan in shared memory, no exchanges: the blocks
//                   are diagonally dominant like A) -- redundantly, so that the inverses are bit-identical everywhere;
//   kry_pre_permute, kry_pre_rows   the own rows of A M^-1, columns regrouped by SZA column, so that the iteration's
//                   product is the same row-times-vector as before with nothing added per step.
__device__ __forceinline__ void post_round_tail(KryState *st, const KryPeers &pe, unsigned long long round, int *sh) {
  const int tid = threadIdx.x;
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    const unsigned int t = atomicAdd(&st->post_tickets, 1u);
    *sh = (t == gridDim.x - 1);
    if (*sh) {
      __threadfence();
      st->post_tickets = 0;
      st->row_queue = 0;
      st->round = round + 1;
    }
  }
  __syncthreads();
  if (*sh && tid < pe.world) st_flag_release(&pe.p[tid]->flag[pe.rank][0], round + 1);
}

__global__ void __launch_bounds__(128)
kry_pre_post(const double *__restrict__ K, int n, const int *__restrict__ rows, int n_rows, double branching, KryWork wk,
             KryPeers pe) {
  __shared__ int sh;
  KryState *st = wk.st;
  const int tid = threadIdx.x;
  const unsigned long long round = st->round;
  for (int r = blockIdx.x; r < n_rows; r += gridDim.x) {
    const int v = rows[r];
    int p0, len;
    pc_block(wk, pc_block_of(wk, pc_perm(wk, v)), &p0, &len);
    if (tid < len) {
      const int e = pc_elem(wk, p0 + tid);
      const double val = (e == v ? 1.0 : 0.0) - branching * K[(size_t) v * n + e];
      for (int q = 0; q < pe.world; q++) st_remote(&pe.p[q]->pre[(size_t) v * KRY_MAX_NR + tid], val);
    }
  }
  __threadfence_system();
  post_round_tail(st, pe, round, &sh);
}

__global__ void __launch_bounds__(KRY_THREADS)
kry_pre_invert(KryWork wk, KryPeers pe) {
  extern __shared__ double Mb[];                   // [nr][nr + 1]
  __shared__ int sh_flag;
  __shared__ double sh_inv;
  KryState *st = wk.st;
  const int tid = threadIdx.x, j = blockIdx.x;
  int p0, nr;
  pc_block(wk, j, &p0, &nr);
  const int ld = nr + 1;
  if (!wait_round(st, pe, st->round, &sh_flag)) return;
  const KryExchange *mine = pe.p[pe.rank];
  for (int e = tid; e < nr * nr; e += KRY_THREADS) {
    const int i = e / nr, c = e - i * nr;
    Mb[i * ld + c] = ld_remote(&mine->pre[(size_t) pc_elem(wk, p0 + i) * KRY_MAX_NR + c]);
  }
  __syncthreads();
  const int tx = tid & 31, ty = tid >> 5;           // thread: columns tx, tx + 32, ...; rows ty, ty + 8, ...
  for (int p = 0; p < nr; p++) {                   // in-place Gauss-Jordan inversion, pivot p
    if (tid == 0) sh_inv = 1.0 / Mb[p * ld + p];
    __syncthreads();
    const double inv = sh_inv;
    for (int c = tid; c < nr; c += KRY_THREADS) Mb[p * ld + c] = (c == p) ? inv : Mb[p * ld + c] * inv;
    __syncthreads();
    double prow[4];                                // this thread's four columns of the pivot row (0 where it must not touch)
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int c = tx + 32 * k;
      prow[k] = (c < nr && c != p) ? Mb[p * ld + c] : 0.0;
    }
#pragma unroll 4
    for (int i = ty; i < nr; i += KRY_WARPS) {
      const double f = (i == p) ? 0.0 : Mb[i * ld + p];
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const int c = tx + 32 * k;
        if (c < nr) Mb[i * ld + c] = fma(-f, prow[k], Mb[i * ld + c]);
      }
    }
    __syncthreads();
    for (int i = tid; i < nr; i += KRY_THREADS)
      if (i != p) Mb[i * ld + p] = -Mb[i * ld + p] * inv;
    __syncthreads();
  }
  double *out = wk.Minv + (size_t) j * wk.run * wk.run;
  for (int e = tid; e < nr * nr; e += KRY_THREADS) out[e] = Mb[(e / nr) * ld + (e % nr)];
}

// own rows of A with the columns in the column order: Bp[r][p] = A[row r][pc_elem(p)]  (a row is read
// once, coalesced, and written once, coalesced; gathering the strided entries inside kry_pre_rows fetched every 64-byte
// line of K eight times: 1.45 ms for the rows of one GPU)
__global__ void __launch_bounds__(KRY_THREADS)
kry_pre_permute(const double *__restrict__ K, int n, const int *__restrict__ rows, int n_rows, double branching, KryWork wk) {
  extern __shared__ double rowbuf[];               // [n]
  const int tid = threadIdx.x;
  for (int r = blockIdx.x; r < n_rows; r += gridDim.x) {
    const int v = rows[r];
    const double *Kr = K + (size_t) v * n;
    for (int c = tid; c < n; c += KRY_THREADS) rowbuf[c] = (c == v ? 1.0 : 0.0) - branching * __ldcs(Kr + c);
    __syncthreads();
    double *out = wk.Bp + (size_t) r * n;
    for (int c = tid; c < n; c += KRY_THREADS) out[c] = rowbuf[pc_elem(wk, c)];
    __syncthreads();
  }
}

constexpr int KRY_PRE_RT = 32;                       // rows of a tile of kry_pre_rows
// Bp[tile rows][block j] <- Bp[tile rows][block j] x Minv_j, in place (a tile is read and written by one CTA only)
__global__ void __launch_bounds__(KRY_THREADS)
kry_pre_rows(int n, int n_rows, KryWork wk) {
  extern __shared__ double sm[];                   // Minv_j [nr][nr] | At [RT][nr]
  const int tid = threadIdx.x, j = blockIdx.x;
  int p0, nr;
  pc_block(wk, j, &p0, &nr);
  double *Mj = sm, *At = sm + nr * nr;
  const double *src = wk.Minv + (size_t) j * wk.run * wk.run;
  for (int e = tid; e < nr * nr; e += KRY_THREADS) Mj[e] = src[e];
  const int cg = tid & 31, rg = tid >> 5;
  // 4 x 4 register tiles: thread (rg, cg) = rows 4 rg .. 4 rg + 3 of the tile, outputs cg, cg + 32, cg + 64, cg + 96 (8 loads
  // from shared memory per 16 FMAs; consecutive threads read consecutive words of Minv: with outputs 4 cg .. 4 cg + 3 the
  // 32-byte stride between threads was an 8-way bank conflict, 28 us per tile instead of 7).  A CTA keeps Minv_j for
  // several row tiles.
  for (int r0 = blockIdx.y * KRY_PRE_RT; r0 < n_rows; r0 += gridDim.y * KRY_PRE_RT) {
    const int rt = min(KRY_PRE_RT, n_rows - r0);
    __syncthreads();                               // (Minv_j in place; the previous tile's At no longer read)
    for (int r = tid >> 5; r < rt; r += KRY_WARPS) {
      const double *in = wk.Bp + (size_t) (r0 + r) * n + p0;
      for (int i = tid & 31; i < nr; i += 32) At[r * nr + i] = in[i];
    }
    __syncthreads();
    double acc[4][4];
#pragma unroll
    for (int u = 0; u < 4; u++)
#pragma unroll
      for (int w = 0; w < 4; w++) acc[u][w] = 0;
    const double *a0 = At + (4 * rg) * nr;
    for (int i = 0; i < nr; i++) {
      double av[4], mv[4];
#pragma unroll
      for (int u = 0; u < 4; u++) av[u] = (4 * rg + u < rt) ? a0[u * nr + i] : 0.0;
#pragma unroll
      for (int w = 0; w < 4; w++) mv[w] = (cg + 32 * w < nr) ? Mj[i * nr + cg + 32 * w] : 0.0;
#pragma unroll
      for (int u = 0; u < 4; u++)
#pragma unroll
        for (int w = 0; w < 4; w++) acc[u][w] = fma(av[u], mv[w], acc[u][w]);
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int r = 4 * rg + u;
      if (r >= rt) continue;
      double *out = wk.Bp + (size_t) (r0 + r) * n + p0;
#pragma unroll
      for (int w = 0; w < 4; w++)
        if (cg + 32 * w < nr) out[cg + 32 * w] = acc[u][w];
    }
  }
}

// =====================================================================================================================
// The whole solve as ONE cooperative launch per rank (kry_loop).  The four launches per step above cost ~36 us of launch
// gaps and cold re-reads around ~5 us of work (measured with events: orth0 8.4, orth1 10.5, orth2 17 us per step on the
// 100x60 grid), which on eight GPUs is six times the product itself.  Here the grid stays resident for the whole
// iteration: every CTA pulls rows for the product; the first ceil(n / 96) CTAs own a slice of the vector and run the two
// Gram-Schmidt passes with three counter barriers among themselves; CTA 0 closes the step (Givens, residual, stop?) and
// publishes the step sequence every CTA waits on.  The same algorithm with the same fixed order of every sum as the launches above
// (the two forms differ in where 1 / |w| multiplies the product, i.e. by rounding).  Everything one CTA reads that another wrote inside the launch goes through L2
// (ld.cg / volatile): L1 is not coherent between SMs.  Every spin loop leaves when st->error is raised (CTA 0 raises it
// when a peer has not posted for 20 s), so a missing rank ends the launch on every rank instead of hanging it.
struct KryLoopArgs {
  const double *K;
  const int *rows;
  const double *S0;
  double *S;
  KryWork wk;
  KryPeers pe;
  double branching, tol;
  int n, n_rows, max_it, orth_blocks;
  bool stage_x;                      // x fits in shared memory beside a grid of at least orth_blocks CTAs
};

__device__ __forceinline__ unsigned int ld_vol_u32(const unsigned int *p) { return *reinterpret_cast<const volatile unsigned int *>(p); }
__device__ __forceinline__ int ld_vol_i32(const int *p) { return *reinterpret_cast<const volatile int *>(p); }

// thread 0: wait until *ctr >= target; false when the solve is being abandoned
__device__ __forceinline__ unsigned int ld_acq_u32(const unsigned int *p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ bool spin_until(const unsigned int *ctr, unsigned int target, KryState *st) {
  unsigned int spins = 0;
  unsigned long long t0 = 0;
  while (ld_acq_u32(ctr) < target) {
    __nanosleep(16);
    if ((++spins & 127u) == 0) {
      if (ld_vol_i32(&st->error)) return false;
      // a barrier of this launch that does not open for 30 s: part of the grid never became resident (another resident
      // grid of another context holds the SMs): give up on every CTA instead of hanging the device
      const unsigned long long t = global_ns();
      if (t0 == 0) t0 = t;
      else if (t - t0 > 30000000000ull) { *reinterpret_cast<volatile int *>(&st->error) = 3; return false; }
    }
  }
  return true;
}
// all threads of every orthogonalising CTA
__device__ __forceinline__ bool orth_barrier(KryState *st, unsigned int target, int *sh_ok) {
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(&st->orth_bar) : "memory");
    *sh_ok = spin_until(&st->orth_bar, target, st) ? 1 : 0;
  }
  __syncthreads();
  return *sh_ok != 0;
}
// all threads of every CTA but CTA 0 (which publishes with step_publish)
// ... and until the orthogonalising CTAs have all arrived `arrivals` times (their slices of w are in place)
__device__ __forceinline__ bool step_wait(KryState *st, unsigned int target, unsigned int arrivals, int *sh_ok) {
  if (threadIdx.x == 0)
    *sh_ok = (spin_until(&st->step_seq, target, st) && spin_until(&st->orth_bar, arrivals, st)) ? 1 : 0;
  __syncthreads();
  return *sh_ok != 0;
}
// an orthogonalising CTA arrives without waiting (the wait is step_wait's)
__device__ __forceinline__ void orth_arrive(KryState *st) {
  __syncthreads();
  if (threadIdx.x == 0) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(&st->orth_bar) : "memory");
}
__device__ __forceinline__ void step_publish(KryState *st, unsigned int value) {
  __syncthreads();
  if (threadIdx.x == 0)
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(&st->step_seq), "r"(value) : "memory");
}
// thread 0 of an orthogonalising CTA: every rank has posted `round` here.  CTA 0 keeps the clock.
__device__ __forceinline__ bool peers_posted(KryState *st, const KryPeers &pe, unsigned long long round, int *sh_ok) {
  if (threadIdx.x == 0) {
    const KryExchange *mine = pe.p[pe.rank];
    const unsigned long long t0 = global_ns();
    int ok = 1;
    for (int q = 0; q < pe.world && ok; q++) {
      unsigned int spins = 0;
      while (ld_flag(&mine->flag[q][0]) < round) {
        __nanosleep(20);
        if ((++spins & 127u) == 0) {
          if (ld_vol_i32(&st->error)) { ok = 0; break; }
          if (blockIdx.x == 0 && global_ns() - t0 > 20000000000ull) {
            *reinterpret_cast<volatile int *>(&st->error) = 1;
            ok = 0;
            break;
          }
        }
      }
    }
    *sh_ok = ok;
  }
  __syncthreads();
  return *sh_ok != 0;
}

// the product phase of a round: MODE as kry_post.  x was written by other CTAs of this launch, so it comes through L2:
// STAGE copies it to shared memory once per round (a CTA with many rows, one GPU), otherwise every row reads it with
// ld.cg beside its row of K (a CTA with one or two rows, eight GPUs: the copy would cost as much as the rows).
// The next row index is requested from the queue while the current row is being multiplied.
constexpr int KRY_UNR = 12;          // loads of K in flight per thread: 5841 / 256 = 22.8 columns per thread = two trips
// PC: the rows are those of A M^-1 (wk.Bp, one per own row slot, columns in the order c' = i_col * nr + i_r), so the
// vector is gathered in that order and the row sum IS the element of the product.
template <int MODE, bool STAGE, bool PC>
__device__ __forceinline__ void loop_post(const KryLoopArgs &a, double *xs, double *red, int *sh_row, unsigned long long round) {
  KryState *st = a.wk.st;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n = a.n;
  const int slot = (int) (round & 1);
  const double *src = MODE == 1 ? (PC ? a.wk.wperm : a.wk.wloc) : a.wk.xsol;
  const double scale = MODE == 1 ? *reinterpret_cast<const volatile double *>(&st->inv_norm) : 1.0;
  constexpr bool WARP_ROWS = STAGE && MODE != 0;   // many rows per CTA: every WARP takes rows from the queue on its own and
                                                   // streams them without a CTA-wide barrier per row (x is in shared memory):
                                                   // product 57 -> 52 us for the 273 MB of one GPU.  (Half rows as work items,
                                                   // to even out the last round, cost more in fences and tickets than they
                                                   // gained: 61 us.)
  if (WARP_ROWS) {
#pragma unroll 8
    for (int c = tid; c < n; c += KRY_THREADS) xs[c] = __ldcg(src + c) * scale;
    __syncthreads();
    for (;;) {
      int slot_row = 0;
      if (lane == 0) slot_row = (int) atomicAdd(&st->row_queue, 1u);
      slot_row = __shfl_sync(0xffffffffu, slot_row, 0);
      if (slot_row >= a.n_rows) break;
      const int i = a.rows[slot_row];
      const double *Kr = PC ? a.wk.Bp + (size_t) slot_row * n : a.K + (size_t) i * n;
      double acc[KRY_UNR];
#pragma unroll
      for (int u = 0; u < KRY_UNR; u++) acc[u] = 0;
      int col = lane;
      for (; col + (KRY_UNR - 1) * 32 < n; col += KRY_UNR * 32) {
        double kk[KRY_UNR];
#pragma unroll
        for (int u = 0; u < KRY_UNR; u++) kk[u] = __ldcs(Kr + col + 32 * u);
#pragma unroll
        for (int u = 0; u < KRY_UNR; u++) acc[u] = fma(kk[u], xs[col + 32 * u], acc[u]);
      }
#pragma unroll
      for (int u = 0; u < KRY_UNR; u++) {
        const int cc = col + 32 * u;
        if (cc < n) acc[u] = fma(__ldcs(Kr + cc), xs[cc], acc[u]);
      }
      double sm = 0;
#pragma unroll
      for (int u = 0; u < KRY_UNR; u++) sm += acc[u];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, o);
      const double val = PC ? sm : xs[i] - a.branching * sm;
      if (lane < a.pe.world) st_remote(&a.pe.p[lane]->w[slot][i], val);
    }
  }
  if (!WARP_ROWS && tid == 0) sh_row[0] = (int) atomicAdd(&st->row_queue, 1u);
  bool staged = false;
  for (int it = 0; !WARP_ROWS; it++) {
    __syncthreads();
    const int slot_row = sh_row[it & 1];
    if (slot_row >= a.n_rows) break;
    if (tid == 0) sh_row[(it + 1) & 1] = (int) atomicAdd(&st->row_queue, 1u);   // in flight during this row
    const int i = a.rows[slot_row];
    double val = 0;
    if (MODE == 0) {
      val = a.S0[i];
    } else {
      if (STAGE && !staged) {
#pragma unroll 8
        for (int c = tid; c < n; c += KRY_THREADS) xs[c] = __ldcg(src + c) * scale;
        staged = true;
        __syncthreads();
      }
      const double *Kr = PC ? a.wk.Bp + (size_t) slot_row * n : a.K + (size_t) i * n;
      double acc[KRY_UNR];
#pragma unroll
      for (int u = 0; u < KRY_UNR; u++) acc[u] = 0;
      int col = tid;
      for (; col + (KRY_UNR - 1) * KRY_THREADS < n; col += KRY_UNR * KRY_THREADS) {
        double kk[KRY_UNR], xx[KRY_UNR];
#pragma unroll
        for (int u = 0; u < KRY_UNR; u++) kk[u] = __ldcs(Kr + col + KRY_THREADS * u);
#pragma unroll
        for (int u = 0; u < KRY_UNR; u++) xx[u] = STAGE ? xs[col + KRY_THREADS * u] : __ldcg(src + col + KRY_THREADS * u);
#pragma unroll
        for (int u = 0; u < KRY_UNR; u++) acc[u] = fma(kk[u], xx[u], acc[u]);
      }
      {
        double kk[KRY_UNR], xx[KRY_UNR];
#pragma unroll
        for (int u = 0; u < KRY_UNR; u++) {
          const int cc = col + KRY_THREADS * u;
          kk[u] = cc < n ? __ldcs(Kr + cc) : 0.0;
          xx[u] = cc < n ? (STAGE ? xs[cc] : __ldcg(src + cc)) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < KRY_UNR; u++) acc[u] = fma(kk[u], xx[u], acc[u]);
      }
      double sm = 0;
#pragma unroll
      for (int u = 0; u < KRY_UNR; u++) sm += acc[u];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, o);
      if (lane == 0) red[warp] = sm;
      __syncthreads();
      if (tid < 32) {
        double t = 0;
#pragma unroll
        for (int k = 0; k < KRY_WARPS; k++) t += red[k];
        if (PC) {
          val = STAGE ? t : scale * t;
        } else {
          const double xi = STAGE ? xs[i] : __ldcg(src + i);
          val = STAGE ? xi - a.branching * t : scale * (xi - a.branching * t);
        }
      }
    }
    if (tid < a.pe.world) st_remote(&a.pe.p[tid]->w[slot][i], val);
  }
  // The threads that stored pieces fence them system-wide (in parallel, once per CTA); when that fence returns the pieces
  // are in the peers' memory, so everything after it -- the ticket, the last CTA's flags -- only has to come later in
  // time.  The last CTA posts the round on all ranks at once, one thread per peer (a release store each): posting them
  // one after the other from one thread cost a round trip over NVLink per peer (measured on eight GPUs: 20 us of a 55 us step).
  if ((WARP_ROWS ? lane : tid) < a.pe.world) __threadfence_system();
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    const unsigned int t = atomicAdd(&st->post_tickets, 1u);
    sh_row[0] = (t == gridDim.x - 1);
    if (sh_row[0]) {
      __threadfence();
      st->post_tickets = 0;
      st->row_queue = 0;
      st->round = round + 1;
    }
  }
  __syncthreads();
  if (sh_row[0] && tid < a.pe.world) {
    if (MODE == 0) st_flag_relaxed(&a.pe.p[tid]->flag[a.pe.rank][1], (unsigned long long) a.n_rows);   // row census, read after the round
    st_flag_release(&a.pe.p[tid]->flag[a.pe.rank][0], round + 1);
  }
  __syncthreads();
}

// partial sums another CTA wrote: through L2
__device__ __forceinline__ void loop_reduce(const double *part, int nv, int n_cta, double *h) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int v0 = warp; v0 < nv; v0 += KRY_VPT * KRY_WARPS) {
    double s[KRY_VPT];
#pragma unroll
    for (int k = 0; k < KRY_VPT; k++) s[k] = 0;
    for (int c0 = 0; c0 < n_cta; c0 += 64) {           // 2 x KRY_VPT loads in flight per lane: one trip to L2 per 64 CTAs
      double lo_[KRY_VPT], hi_[KRY_VPT];
#pragma unroll
      for (int k = 0; k < KRY_VPT; k++) {
        const double *p = part + (size_t) min(v0 + k * KRY_WARPS, nv - 1) * KRY_MAX_B + c0;
        lo_[k] = (c0 + lane < n_cta) ? __ldcg(p + lane) : 0.0;
        hi_[k] = (c0 + 32 + lane < n_cta) ? __ldcg(p + 32 + lane) : 0.0;
      }
#pragma unroll
      for (int k = 0; k < KRY_VPT; k++) { s[k] += lo_[k]; s[k] += hi_[k]; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int k = 0; k < KRY_VPT; k++) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
#pragma unroll
    for (int k = 0; k < KRY_VPT; k++)
      if (lane == 0 && v0 + k * KRY_WARPS < nv) h[v0 + k * KRY_WARPS] = s[k];
  }
}
__device__ __forceinline__ double loop_sum_partials(const double *p, int n_cta) {   // a warp; as warp_sum_partials, through L2
  const int lane = threadIdx.x & 31;
  double s = 0;
  for (int c = lane; c < n_cta; c += 32) s += __ldcg(p + c);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  return s;
}

__global__ void __launch_bounds__(KRY_THREADS)
kry_loop(KryLoopArgs a) {
  extern __shared__ double xs[];
  __shared__ double ws[KRY_SLICE];
  __shared__ double red[KRY_WARPS][KRY_SLICE];
  __shared__ double h[KRY_MAX_IT + 2], hsum[KRY_MAX_IT + 2];
  __shared__ double rot[2 * KRY_MAX_IT + 2], gs[KRY_MAX_IT + 2];      // CTA 0: the rotations and the rotated right-hand side
  __shared__ double scratch[KRY_WARPS];
  __shared__ double sh_val;
  __shared__ int sh_flag, sh_row[2];
  KryState *st = a.wk.st;
  const KryWork &wk = a.wk;
  const KryPeers &pe = a.pe;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n = a.n;
  const int cta = blockIdx.x, n_orth = a.orth_blocks;
  const bool orth = cta < n_orth;
  const int lo = cta * KRY_SLICE, len = orth ? min(KRY_SLICE, n - lo) : 0;
  unsigned long long round = st->round;          // every CTA counts the rounds itself (st->round is for the host)
  unsigned int bar = 0, seq = 0;
  const KryExchange *mine = pe.p[pe.rank];
  const bool stage = a.stage_x && a.n_rows > 3 * (int) gridDim.x;   // rows per CTA and round
  const bool pc = wk.run > 0;                          // right-preconditioned: the iteration is on u, S = M^-1 u
  int pos_perm = 0;                                    // where this thread's element of the slice sits in the column order of Bp
  if (pc && tid < len) pos_perm = pc_perm(wk, lo + tid);
  const bool clock = cta == 0 && tid == 0;
  unsigned long long t_mark = 0, t_sub = 0, t_acc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};

  // ---- round 0: the right-hand side, assembled from every rank's own rows
  loop_post<0, false, false>(a, xs, &red[0][0], sh_row, round);
  round++;
  double beta = 0;
  ++bar;                                           // (every CTA counts the barriers of the orthogonalising ones)
  if (orth) {
    if (!peers_posted(st, pe, round, &sh_flag)) return;
    const int slot = (int) ((round - 1) & 1);
    double b = 0;
    if (tid < len) {
      b = ld_remote(&mine->w[slot][lo + tid]);
      wk.bvec[lo + tid] = b;
      wk.wloc[lo + tid] = b;
      if (pc) wk.wperm[pos_perm] = b;
      ws[tid] = b;
    }
    const double s2 = slice_sum(b * b, scratch);
    if (tid == 0) wk.npart[cta] = s2;
    if (!orth_barrier(st, bar * n_orth, &sh_flag)) return;
    if (warp == 0) {
      const double t = loop_sum_partials(wk.npart, n_orth);
      if (lane == 0) sh_val = t;
    }
    __syncthreads();
    beta = sqrt(sh_val);
    const double inv = beta > 0 ? 1.0 / beta : 0.0;
    if (tid < len) wk.V[lo + tid] = ws[tid] * inv;                 // basis vector 0, this CTA's slice (read only by this CTA)
    if (cta == 0 && tid == 0) {
      unsigned long long census = 0;
      for (int q = 0; q < pe.world; q++) census += ld_flag(&mine->flag[q][1]);
      st->beta = beta;
      st->inv_norm = inv;
      gs[0] = beta;
      st->iter = 0;
      st->res = 1.0;
      st->true_res = -1.0;
      st->converged = beta > 0 ? 0 : 1;
      int stop = beta > 0 ? 0 : 1;
      if (census != (unsigned long long) n) { st->error = 2; stop = 1; }
      st->done = stop;
    }
  }
  ++seq;
  if (cta == 0) step_publish(st, seq);
  if (!step_wait(st, seq, bar * n_orth, &sh_flag)) return;
  if (ld_vol_i32(&st->error)) return;
  int done = ld_vol_i32(&st->done);

  // ---- Arnoldi steps
  int j = 0;
  while (!done) {
    if (clock) t_mark = global_ns();
    if (pc) {
      if (stage) loop_post<1, true, true>(a, xs, &red[0][0], sh_row, round);
      else loop_post<1, false, true>(a, xs, &red[0][0], sh_row, round);
    } else {
      if (stage) loop_post<1, true, false>(a, xs, &red[0][0], sh_row, round);
      else loop_post<1, false, false>(a, xs, &red[0][0], sh_row, round);
    }
    round++;
    bar += 3;
    if (orth) {
      const int nv = j + 1;
      if (clock) { const unsigned long long t = global_ns(); t_acc[0] += t - t_mark; t_mark = t; }
      if (!peers_posted(st, pe, round, &sh_flag)) return;
      if (clock) { const unsigned long long t = global_ns(); t_acc[1] += t - t_mark; t_mark = t; t_sub = t; }
      const int slot = (int) ((round - 1) & 1);
      if (tid < len) ws[tid] = ld_remote(&mine->w[slot][lo + tid]);
      __syncthreads();
      slice_dots(ws, wk, lo, len, nv, wk.part1);
      if (clock) { const unsigned long long t = global_ns(); t_acc[4] += t - t_sub; t_sub = t; }
      if (!orth_barrier(st, (bar - 2) * n_orth, &sh_flag)) return;
      if (clock) { const unsigned long long t = global_ns(); t_acc[5] += t - t_sub; t_sub = t; }
      loop_reduce(wk.part1, nv, n_orth, h);
      __syncthreads();
      for (int v = tid; v < nv; v += KRY_THREADS) hsum[v] = h[v];
      slice_update(ws, wk, lo, len, nv, h, red, -1.0);
      slice_dots(ws, wk, lo, len, nv, wk.part2);
      {   // |w1|^2 of the slice rides with the second pass's partials (row nv): after the second pass
          // |w|^2 = |w1|^2 - sum h2^2 (h2 is a re-orthogonalisation: tiny against |w1|, no cancellation), so the norm
          // needs no reduction -- and no barrier -- of its own
        const double w1 = slice_sum(tid < len ? ws[tid] * ws[tid] : 0.0, scratch);
        if (tid == 0) wk.part2[(size_t) nv * KRY_MAX_B + cta] = w1;
      }
      if (clock) { const unsigned long long t = global_ns(); t_acc[6] += t - t_sub; t_sub = t; }
      if (!orth_barrier(st, (bar - 1) * n_orth, &sh_flag)) return;
      if (clock) { const unsigned long long t = global_ns(); t_acc[7] += t - t_sub; t_sub = t; }
      loop_reduce(wk.part2, nv + 1, n_orth, h);
      __syncthreads();
      for (int v = tid; v < nv; v += KRY_THREADS) hsum[v] += h[v];
      if (warp == 0) {
        double q = 0;
        for (int v = lane; v < nv; v += 32) q = fma(h[v], h[v], q);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
        if (lane == 0) sh_val = fmax(h[nv] - q, 0.0);
      }
      slice_update(ws, wk, lo, len, nv, h, red, -1.0);       // (its barriers publish sh_val)
      if (tid < len) {                                             // unnormalised: the product scales by 1 / |w|
        if (pc) wk.wperm[pos_perm] = ws[tid];
        else wk.wloc[lo + tid] = ws[tid];
      }
      if (clock) { const unsigned long long t = global_ns(); t_acc[8] += t - t_sub; t_sub = t; }
      // the slices of w must be in place before the next product reads them: arrive here, wait with everyone at the end
      // of the step (CTA 0 closes the step meanwhile)
      orth_arrive(st);
      const double hn = sqrt(sh_val);
      const double inv = hn > 0 ? 1.0 / hn : 0.0;
      if (tid < len) wk.V[(size_t) (j + 1) * wk.ns + lo + tid] = ws[tid] * inv;
      if (clock) { const unsigned long long t = global_ns(); t_acc[2] += t - t_mark; t_mark = t; }
      if (cta == 0) {
        if (tid == 0) {
          double hi = hsum[0];
          for (int i = 0; i < j; i++) {
            const double c_ = rot[2 * i], s_ = rot[2 * i + 1], up = hsum[i + 1];
            hsum[i] = c_ * hi + s_ * up;
            hi = -s_ * hi + c_ * up;
          }
          const double d = hypot(hi, hn);
          const double c_ = d > 0 ? hi / d : 1.0, s_ = d > 0 ? hn / d : 0.0;
          hsum[j] = d;
          rot[2 * j] = c_; rot[2 * j + 1] = s_;
          const double gj = gs[j];
          gs[j + 1] = -s_ * gj;
          gs[j] = c_ * gj;
          const double res = fabs(gs[j + 1]) / beta;
          st->res = res;
          st->iter = j + 1;
          st->inv_norm = inv;
          const bool conv = res <= a.tol || hn == 0.0;
          st->converged = conv ? 1 : 0;
          st->done = (conv || j + 1 >= a.max_it) ? 1 : 0;
        }
        __syncthreads();
        for (int i = tid; i <= j; i += KRY_THREADS) wk.R[(size_t) i * KRY_MAX_IT + j] = hsum[i];
        if (clock) { const unsigned long long t = global_ns(); t_acc[3] += t - t_mark; t_mark = t; }
      }
    }
    ++seq;
    if (cta == 0) step_publish(st, seq);
    if (clock) t_sub = global_ns();
    if (!step_wait(st, seq, bar * n_orth, &sh_flag)) return;
    if (clock) t_acc[9] += global_ns() - t_sub;
    done = ld_vol_i32(&st->done);
    j++;
  }
  if (ld_vol_i32(&st->error)) return;
  if (clock)
    for (int q = 0; q < 10; q++) st->t_phase[q] = t_acc[q];

  // ---- S = V y, y = R^-1 g: CTA 0 substitutes (row l on thread l), the slices combine
  const int k = j;                                 // Arnoldi steps taken (0 when S0 = 0)
  if (cta == 0) {
    double gl = tid < k ? gs[tid] : 0.0;
    for (int i = k - 1; i >= 0; i--) {
      if (tid == i) {
        const double y = gl / wk.R[(size_t) i * KRY_MAX_IT + i];
        sh_val = y;
        wk.y[i] = y;
      }
      __syncthreads();
      if (tid < i) gl -= wk.R[(size_t) tid * KRY_MAX_IT + i] * sh_val;
      __syncthreads();
    }
  }
  ++seq;
  if (cta == 0) step_publish(st, seq);
  if (!step_wait(st, seq, bar * n_orth, &sh_flag)) return;
  ++bar;
  if (orth) {
    for (int v = tid; v < k; v += KRY_THREADS) h[v] = __ldcg(wk.y + v);
    if (tid < KRY_SLICE) ws[tid] = 0;
    __syncthreads();
    slice_update(ws, wk, lo, len, k, h, red, 1.0);
    if (!pc) {
      if (tid < len) { wk.xsol[lo + tid] = ws[tid]; a.S[lo + tid] = ws[tid]; }
    } else if (tid < len) {
      wk.usol[lo + tid] = ws[tid];
    }
    orth_arrive(st);
  }
  ++seq;
  if (cta == 0) step_publish(st, seq);
  if (!step_wait(st, seq, bar * n_orth, &sh_flag)) return;
  if (pc) {                                        // S = M^-1 u, block by block: unknown at position p0 + i of block b =
    ++bar;                                         // row i of Minv_b . u[unknowns of block b]
    if (orth) {
      for (int e = warp; e < len; e += KRY_WARPS) {
        const int v = lo + e, p = pc_perm(wk, v), b = pc_block_of(wk, p);
        int p0, nr;
        pc_block(wk, b, &p0, &nr);
        const double *mrow = wk.Minv + (size_t) b * wk.run * wk.run + (size_t) (p - p0) * nr;
        double sum = 0;
        for (int i = lane; i < nr; i += 32) sum = fma(mrow[i], __ldcg(wk.usol + pc_elem(wk, p0 + i)), sum);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if (lane == 0) { wk.xsol[v] = sum; a.S[v] = sum; }
      }
      orth_arrive(st);
    }
    ++seq;
    if (cta == 0) step_publish(st, seq);
    if (!step_wait(st, seq, bar * n_orth, &sh_flag)) return;
  }

  // ---- the true residual: one more product, with the solution
  if (stage) loop_post<2, true, false>(a, xs, &red[0][0], sh_row, round);
  else loop_post<2, false, false>(a, xs, &red[0][0], sh_row, round);
  round++;
  if (orth) {
    if (!peers_posted(st, pe, round, &sh_flag)) return;
    const int slot = (int) ((round - 1) & 1);
    double r = 0;
    if (tid < len) r = wk.bvec[lo + tid] - ld_remote(&mine->w[slot][lo + tid]);
    const double s2 = slice_sum(r * r, scratch);
    if (tid == 0) wk.npart[cta] = s2;
    if (!orth_barrier(st, ++bar * n_orth, &sh_flag)) return;     // (the last barrier: only these CTAs count it)
    if (cta == 0 && warp == 0) {
      const double t = loop_sum_partials(wk.npart, n_orth);
      if (lane == 0) st->true_res = beta > 0 ? sqrt(t) / beta : 0.0;
    }
  }
}

// =====================================================================================================================
// The adjoint system (I - w K)^T lambda = r runs through the machinery above unchanged, on K^T: the preconditioner's
// set-up then builds the diagonal blocks of A^T (= M^T), their inverses and the rows of A^T M^-T, kry_loop iterates with
// the tuned row product, and its true-residual pass checks the adjoint system itself.  (A column-wise product inside
// kry_loop would have to reduce full-length partial vectors in every step.)  Kt = K^T, n x n row major, through padded
// 32 x 32 tiles in shared memory: reads and writes are rows of 256 bytes, K streams through L2 with evict-first loads
// (273 MB on the 100x60 grid, more than L2 holds).  The padding keeps both tile accesses free of bank conflicts (a double
// spans two banks; a warp's 256 bytes go out as two half-warp phases).
constexpr int KT_TILE = 32, KT_ROWS = 8;
__global__ void __launch_bounds__(KT_TILE * KT_ROWS)
kry_transpose(const double *__restrict__ K, int n, double *__restrict__ Kt) {
  __shared__ double tile[KT_TILE][KT_TILE + 1];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int c0 = blockIdx.x * KT_TILE, r0 = blockIdx.y * KT_TILE;
  double v[KT_TILE / KT_ROWS];
#pragma unroll
  for (int k = 0; k < KT_TILE / KT_ROWS; k++) {
    const int r = r0 + ty + k * KT_ROWS, col = c0 + tx;
    v[k] = (r < n && col < n) ? __ldcs(K + (size_t) r * n + col) : 0.0;
  }
#pragma unroll
  for (int k = 0; k < KT_TILE / KT_ROWS; k++) tile[ty + k * KT_ROWS][tx] = v[k];
  __syncthreads();
#pragma unroll
  for (int k = 0; k < KT_TILE / KT_ROWS; k++) {
    const int r = c0 + ty + k * KT_ROWS, col = r0 + tx;     // row r of Kt = column r of K
    if (r < n && col < n) Kt[(size_t) r * n + col] = tile[tx][ty + k * KT_ROWS];
  }
}

size_t carve_bytes(size_t &off, size_t bytes) {
  off = (off + 255) & ~size_t(255);
  const size_t at = off;
  off += bytes;
  return at;
}

// One rank's GMRES over a fixed set of rows, for one system after another (the forward solve: every emission; the
// adjoint: every right-hand side).  kry_open carves the work area and uploads the rows; kry_setup builds the
// preconditioner of one matrix (K, branching); kry_iterate launches the iteration for one right-hand side into one
// solution vector.  No iteration launch writes what kry_setup wrote (Minv and Bp of the work area, pre[] of the exchange
// blocks): one set-up serves any number of right-hand sides.
struct KrySolver {
  KryWork wk;
  KryPeers pe;
  int *d_rows;
  int n, n_rows, cta_cap;
  bool pc, fused;                    // fused: the one-launch form (B200RT_KRYLOV_FUSED=0: the per-step launches)
  int pc_run, pc_blocks;
  double tol;
  int max_it, post_blocks, orth_blocks;
  KryState *h_st;                    // page-locked: [0, 63) the per-step form's chunk read-backs, [63 + k] final state k
  bool trace;                        // B200RT_KRYLOV_TRACE=1: event marks around the set-up and the first 48 steps
  std::vector<cudaEvent_t> marks;
};

// work: this solver's work area; round_base: the round counter its exchange blocks have reached (restored when the work
// area is new); n_final: final states the caller reads back
int kry_open(b200rt_ctx *c, const std::vector<int> &rows, int n, int nu, DevBuf &work, unsigned long long round_base,
             void *const *blocks, int rank, int world, int cta_cap, int n_final, KrySolver &ks) {
  const int n_rows = (int) rows.size();
  const int ns = (n + 31) & ~31;
  size_t off = 0;
  const size_t o_st = carve_bytes(off, sizeof(KryState));
  const size_t o_V = carve_bytes(off, (size_t) (KRY_MAX_IT + 1) * ns * sizeof(double));
  const size_t o_w = carve_bytes(off, (size_t) ns * sizeof(double)), o_b = carve_bytes(off, (size_t) ns * sizeof(double)),
               o_x = carve_bytes(off, (size_t) ns * sizeof(double));
  const size_t o_p1 = carve_bytes(off, (size_t) (KRY_MAX_IT + 1) * KRY_MAX_B * sizeof(double)),
               o_p2 = carve_bytes(off, (size_t) (KRY_MAX_IT + 1) * KRY_MAX_B * sizeof(double));
  const size_t o_np = carve_bytes(off, KRY_MAX_B * sizeof(double));
  const size_t o_R = carve_bytes(off, (size_t) (KRY_MAX_IT + 1) * KRY_MAX_IT * sizeof(double));
  const size_t o_cs = carve_bytes(off, (KRY_MAX_IT + 1) * sizeof(double)), o_sn = carve_bytes(off, (KRY_MAX_IT + 1) * sizeof(double)),
               o_g = carve_bytes(off, (KRY_MAX_IT + 1) * sizeof(double)), o_y = carve_bytes(off, (KRY_MAX_IT + 1) * sizeof(double));
  const size_t o_rows = carve_bytes(off, (size_t) std::max(n, 1) * sizeof(int));
  // right preconditioner over the SZA columns (spherical grids; B200RT_KRYLOV_PC=0 switches it off): every column is cut,
  // from the lowest voxel up, into runs of KRY_MAX_NR / nu radial voxels with all their states (KryWork); runs as equal
  // as whole voxels allow took as many or more steps (tests/krylov_multiplet_model.py, pc_blocks)
  const int pc_nr = c->hg.n_rb - 1, pc_nc = c->hg.n_sb - 1;
  bool pc = !c->hg.pp && pc_nr >= 2 && pc_nc >= 2 && pc_nr * pc_nc == c->hg.n_vox && nu <= KRY_MAX_NR;
  if (const char *env = getenv("B200RT_KRYLOV_PC")) pc = pc && atoi(env) != 0;
  if (const char *env = getenv("B200RT_KRYLOV_FUSED")) pc = pc && atoi(env) != 0;     // the per-step launches iterate on A itself
  int pc_runs = 1, pc_run = 0;
  if (pc) {
    const int run_vox = std::min(pc_nr, KRY_MAX_NR / nu);
    pc_run = nu * run_vox;
    pc_runs = (pc_nr + run_vox - 1) / run_vox;
  }
  const int pc_blocks = pc_nc * pc_runs;
  const size_t o_usol = carve_bytes(off, (size_t) ns * sizeof(double)), o_wperm = carve_bytes(off, (size_t) ns * sizeof(double));
  const size_t o_minv = carve_bytes(off, pc ? (size_t) pc_blocks * pc_run * pc_run * sizeof(double) : 16);
  const bool fresh = work.bytes < off;
  B200RT_CUDA(c, work.ensure(off));
  char *base = static_cast<char *>(work.p);
  if (fresh) {    // the round counter lives with the exchange block's life: it restarts only together with it
    B200RT_CUDA(c, cudaMemsetAsync(base + o_st, 0, sizeof(KryState), c->stream));
    if (round_base) {
      B200RT_CUDA(c, cudaMemcpyAsync(base + o_st, &round_base, sizeof(unsigned long long), cudaMemcpyHostToDevice, c->stream));
      B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
    }
  }
  KryWork &wk = ks.wk;
  wk.st = reinterpret_cast<KryState *>(base + o_st);
  wk.V = reinterpret_cast<double *>(base + o_V);
  wk.wloc = reinterpret_cast<double *>(base + o_w); wk.bvec = reinterpret_cast<double *>(base + o_b);
  wk.xsol = reinterpret_cast<double *>(base + o_x);
  wk.part1 = reinterpret_cast<double *>(base + o_p1); wk.part2 = reinterpret_cast<double *>(base + o_p2);
  wk.npart = reinterpret_cast<double *>(base + o_np);
  wk.R = reinterpret_cast<double *>(base + o_R);
  wk.cs = reinterpret_cast<double *>(base + o_cs); wk.sn = reinterpret_cast<double *>(base + o_sn);
  wk.g = reinterpret_cast<double *>(base + o_g); wk.y = reinterpret_cast<double *>(base + o_y);
  wk.ns = ns;
  wk.usol = reinterpret_cast<double *>(base + o_usol);
  wk.wperm = reinterpret_cast<double *>(base + o_wperm);
  wk.Minv = reinterpret_cast<double *>(base + o_minv);
  wk.Bp = nullptr;
  wk.run = 0; wk.n_col = pc_nc; wk.nu = nu; wk.cl = pc_nr * nu; wk.n_runs = pc_runs;
  if (pc) {       // (shared by the forward and the adjoint solver: every set-up rewrites each row an iteration reads)
    B200RT_CUDA(c, c->kry_bp.ensure((size_t) std::max(n_rows, 1) * n * sizeof(double)));
    wk.Bp = c->kry_bp.as<double>();
  }
  ks.d_rows = reinterpret_cast<int *>(base + o_rows);
  B200RT_CUDA(c, c->host_stage.ensure((size_t) std::max(n, 1) * sizeof(int)));
  std::memcpy(c->host_stage.p, rows.data(), (size_t) n_rows * sizeof(int));
  B200RT_CUDA(c, cudaMemcpyAsync(ks.d_rows, c->host_stage.p, (size_t) n_rows * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  for (int q = 0; q < KRY_MAX_WORLD; q++) ks.pe.p[q] = q < world ? static_cast<KryExchange *>(blocks[q]) : nullptr;
  ks.pe.rank = rank; ks.pe.world = world;

  ks.tol = 1e-13;
  if (const char *env = getenv("B200RT_KRYLOV_TOL")) ks.tol = atof(env);
  ks.max_it = KRY_MAX_IT;
  if (const char *env = getenv("B200RT_KRYLOV_MAXIT")) ks.max_it = std::max(1, std::min(KRY_MAX_IT, atoi(env)));
  ks.fused = true;
  if (const char *env = getenv("B200RT_KRYLOV_FUSED")) ks.fused = atoi(env) != 0;

  ks.n = n; ks.n_rows = n_rows; ks.cta_cap = cta_cap;
  ks.pc = pc; ks.pc_run = pc_run; ks.pc_blocks = pc_blocks;
  ks.post_blocks = std::max(1, std::min(n_rows, NUM_SMS * 8));   // CTAs pull rows from a queue
  ks.orth_blocks = (n + KRY_SLICE - 1) / KRY_SLICE;
  B200RT_CUDA(c, c->host_scratch.ensure((63 + (size_t) std::max(n_final, 1)) * sizeof(KryState)));
  ks.h_st = c->host_scratch.as<KryState>();
  static const bool trace = getenv("B200RT_KRYLOV_TRACE") != nullptr;
  ks.trace = trace;
  ks.marks.clear();
  return B200RT_OK;
}

// everything but the round counter starts from zero (no kernel of this solver is in flight here)
cudaError_t kry_reset(const KrySolver &ks, cudaStream_t s) {
  return cudaMemsetAsync(reinterpret_cast<char *>(ks.wk.st) + offsetof(KryState, iter), 0,
                         sizeof(KryState) - offsetof(KryState, iter), s);
}

void kry_mark(KrySolver &ks, cudaStream_t s) {
  cudaEvent_t ev;
  cudaEventCreate(&ev);
  cudaEventRecord(ev, s);
  ks.marks.push_back(ev);
}

// the preconditioner of the one-launch form: block entries to all ranks, inverses, rows of A M^-1
int kry_setup(b200rt_ctx *c, KrySolver &ks, const double *K, double branching, int *launches) {
  if (!(ks.fused && ks.pc)) return B200RT_OK;
  KryWork &wk = ks.wk;
  const int n = ks.n, n_rows = ks.n_rows, pc_run = ks.pc_run, pc_blocks = ks.pc_blocks;
  cudaStream_t s = c->stream;
  wk.run = pc_run;
  const size_t sm_inv = (size_t) pc_run * (pc_run + 1) * sizeof(double);
  const size_t sm_rows = ((size_t) pc_run * pc_run + (size_t) KRY_PRE_RT * pc_run) * sizeof(double);
  B200RT_CUDA(c, cudaFuncSetAttribute(kry_pre_invert, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) sm_inv));
  B200RT_CUDA(c, cudaFuncSetAttribute(kry_pre_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) sm_rows));
  B200RT_CUDA(c, cudaFuncSetAttribute(kry_pre_permute, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ((size_t) n * sizeof(double))));
  if (ks.trace) kry_mark(ks, s);
  kry_pre_post<<<std::max(1, std::min(n_rows, 4 * NUM_SMS)), 128, 0, s>>>(K, n, ks.d_rows, n_rows, branching, wk, ks.pe);
  if (ks.trace) kry_mark(ks, s);
  kry_pre_invert<<<pc_blocks, KRY_THREADS, sm_inv, s>>>(wk, ks.pe);
  if (ks.trace) kry_mark(ks, s);
  if (n_rows > 0) {
    kry_pre_permute<<<std::min(n_rows, 4 * NUM_SMS), KRY_THREADS, (size_t) n * sizeof(double), s>>>(K, n, ks.d_rows, n_rows, branching, wk);
    kry_pre_rows<<<dim3(pc_blocks, std::max(1, std::min((n_rows + KRY_PRE_RT - 1) / KRY_PRE_RT, 2 * NUM_SMS / pc_blocks))), KRY_THREADS, sm_rows, s>>>(n, n_rows, wk);
  }
  if (ks.trace) kry_mark(ks, s);
  *launches += 4;
  return B200RT_OK;
}

// one iteration for the right-hand side S0 into S: the one-launch form, or the per-step launches when the cooperative
// grid does not fit (or B200RT_KRYLOV_FUSED=0); *fused says which ran
int kry_iterate(b200rt_ctx *c, KrySolver &ks, const double *K, double branching, const double *S0, double *S,
                int *launches, bool *fused_out) {
  KryWork wk = ks.wk;
  const KryPeers &pe = ks.pe;
  const int n = ks.n, n_rows = ks.n_rows, orth_blocks = ks.orth_blocks, post_blocks = ks.post_blocks, max_it = ks.max_it;
  const int *d_rows = ks.d_rows;
  KryState *h_st = ks.h_st;
  cudaStream_t s = c->stream;
  constexpr int CHUNK = 16;
  bool fused = ks.fused;
  if (fused) {
    // x staged in shared memory (n * 8 bytes per CTA) where that leaves room for a grid of orth_blocks CTAs; otherwise
    // (above ~14k unknowns on a B200) the rows read x through L2 and the CTAs need no dynamic shared memory
    int cap = ks.cta_cap > 0 ? ks.cta_cap : 3 * NUM_SMS;
    if (const char *env = getenv("B200RT_KRYLOV_CTAS")) cap = std::max(1, atoi(env));
    int grid = 0;
    size_t smem = 0;
    for (const size_t try_smem : {(size_t) n * sizeof(double), (size_t) 0}) {
      int per_sm = 0;
      cudaError_t e_occ = cudaFuncSetAttribute(kry_loop, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) try_smem);
      if (e_occ == cudaSuccess) e_occ = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kry_loop, KRY_THREADS, try_smem);
      if (e_occ != cudaSuccess) { cudaGetLastError(); continue; }
      grid = std::min(cap, per_sm * NUM_SMS);
      smem = try_smem;
      if (grid >= orth_blocks) break;
    }
    if (grid < orth_blocks) {
      fused = false;                             // (a grid too small to own every slice of the vector: the launches below)
    } else {
      KryLoopArgs a;
      a.K = K; a.rows = d_rows; a.S0 = S0; a.S = S; a.wk = wk; a.pe = pe;
      a.branching = branching; a.tol = ks.tol; a.n = n; a.n_rows = n_rows; a.max_it = max_it; a.orth_blocks = orth_blocks;
      a.stage_x = smem > 0;
      void *kargs[] = {&a};
      const cudaError_t e_l = cudaLaunchCooperativeKernel((void *) kry_loop, dim3(grid), dim3(KRY_THREADS), kargs, smem, s);
      if (e_l == cudaSuccess) *launches += 1;
      else { cudaGetLastError(); fused = false; }
    }
  }
  *fused_out = fused;
  if (fused) return B200RT_OK;
  wk.run = 0;                                      // (the launches below iterate on A itself)
  kry_post<0><<<post_blocks, KRY_THREADS, 0, s>>>(K, n, d_rows, n_rows, branching, S0, wk, pe);
  kry_begin<<<orth_blocks, KRY_THREADS, 0, s>>>(n, wk, pe, ks.tol, max_it);
  *launches += 2;
  // Arnoldi steps in chunks; the state after chunk k is read back while chunk k + 1 runs, so at most two chunks of
  // (empty: every kernel returns at once after `done`) launches follow the step that converged
  const int n_chunks = (max_it + CHUNK - 1) / CHUNK;
  std::vector<cudaEvent_t> read(n_chunks);
  bool stop = false;
  for (int k = 0; k < n_chunks && !stop; k++) {
    for (int it = 0; it < CHUNK && k * CHUNK + it < max_it; it++) {
      const bool tr = ks.trace && k * CHUNK + it < 48;
      if (tr) kry_mark(ks, s);
      kry_post<1><<<post_blocks, KRY_THREADS, 0, s>>>(K, n, d_rows, n_rows, branching, S0, wk, pe);
      if (tr) kry_mark(ks, s);
      kry_orth<0><<<orth_blocks, KRY_THREADS, 0, s>>>(n, wk, pe);
      if (tr) kry_mark(ks, s);
      kry_orth<1><<<orth_blocks, KRY_THREADS, 0, s>>>(n, wk, pe);
      if (tr) kry_mark(ks, s);
      kry_orth<2><<<orth_blocks, KRY_THREADS, 0, s>>>(n, wk, pe);
      if (tr) kry_mark(ks, s);
      *launches += 4;
    }
    B200RT_CUDA(c, cudaMemcpyAsync(h_st + k, wk.st, sizeof(KryState), cudaMemcpyDeviceToHost, s));
    read[k] = api::PhaseTimer::take(c);
    B200RT_CUDA(c, cudaEventRecord(read[k], s));
    if (k >= 1) {
      B200RT_CUDA(c, cudaEventSynchronize(read[k - 1]));
      stop = h_st[k - 1].done != 0;
    }
  }
  kry_backsolve<<<1, 32, 0, s>>>(wk);
  kry_solution<<<orth_blocks, KRY_THREADS, 0, s>>>(n, wk, S);
  kry_post<2><<<post_blocks, KRY_THREADS, 0, s>>>(K, n, d_rows, n_rows, branching, S0, wk, pe);
  kry_residual<<<orth_blocks, KRY_THREADS, 0, s>>>(n, wk, pe);
  *launches += 4;
  return B200RT_OK;
}

// B200RT_KRYLOV_TRACE: what the marks of the last set-up and iteration measured (after the stream has been synchronised)
void kry_trace_report(KrySolver &ks, bool fused, const KryState &fin) {
  if (!ks.trace) return;
  auto &marks = ks.marks;
  if (fused && marks.size() == 4) {
    float ms[3];
    for (int q = 0; q < 3; q++) cudaEventElapsedTime(&ms[q], marks[q], marks[q + 1]);
    fprintf(stderr, "krylov trace: preconditioner set-up [us]: block entries to all ranks %.1f  inverses %.1f  rows of A M^-1 %.1f\n",
            ms[0] * 1e3, ms[1] * 1e3, ms[2] * 1e3);
    for (auto ev : marks) cudaEventDestroy(ev);
    marks.clear();
  }
  if (!marks.empty()) {
    double sum[4] = {0, 0, 0, 0};
    const int steps_traced = (int) marks.size() / 5;
    for (int st_ = 0; st_ < steps_traced; st_++)
      for (int q = 0; q < 4; q++) {
        float ms = 0;
        cudaEventElapsedTime(&ms, marks[st_ * 5 + q], marks[st_ * 5 + q + 1]);
        sum[q] += ms;
      }
    fprintf(stderr, "krylov trace (%d steps, us per step): post %.2f  orth0 %.2f  orth1 %.2f  orth2 %.2f\n", steps_traced,
            sum[0] / steps_traced * 1e3, sum[1] / steps_traced * 1e3, sum[2] / steps_traced * 1e3, sum[3] / steps_traced * 1e3);
    for (auto ev : marks) cudaEventDestroy(ev);
    marks.clear();
  }
  if (fused && fin.iter > 0)
    fprintf(stderr, "krylov trace (one launch, %d steps, CTA 0's clock, us per step): product %.2f  wait for peers %.2f  "
            "orthogonalisation %.2f (pass / barrier: %.2f / %.2f, %.2f / %.2f, %.2f / %.2f)  closing %.2f\n", fin.iter,
            fin.t_phase[0] * 1e-3 / fin.iter, fin.t_phase[1] * 1e-3 / fin.iter, fin.t_phase[2] * 1e-3 / fin.iter,
            fin.t_phase[4] * 1e-3 / fin.iter, fin.t_phase[5] * 1e-3 / fin.iter, fin.t_phase[6] * 1e-3 / fin.iter,
            fin.t_phase[7] * 1e-3 / fin.iter, fin.t_phase[8] * 1e-3 / fin.iter, fin.t_phase[9] * 1e-3 / fin.iter,
            fin.t_phase[3] * 1e-3 / fin.iter);
}

// the outcome of one iteration; `who` names the entry point, `hint` follows a residual that did not converge
int kry_status(b200rt_ctx *c, const KryState &fin, const std::string &who, const char *hint) {
  if (fin.error == 3)
    return fail(c, B200RT_ERR_CUDA, who + ": the resident grid of the solve never became complete (30 s): another resident "
                                          "grid on this device holds its SMs (B200RT_KRYLOV_CTAS limits the grid; B200RT_KRYLOV_FUSED=0 avoids it)");
  if (fin.error == 2)
    return fail(c, B200RT_ERR_STATE, who + ": the rows the ranks built do not add up to the grid (every voxel must be in exactly one rank's influence call)");
  if (fin.error)
    return fail(c, B200RT_ERR_CUDA, who + ": a peer never posted its rows (20 s): all ranks must call it, with the same grid");
  if (!fin.converged)
    return fail(c, B200RT_ERR_NOT_DOMINANT, who + ": GMRES residual " + std::to_string(fin.res) + " after " +
                                                std::to_string(fin.iter) + " steps" + hint);
  if (!(fin.true_res <= 1e-8))
    return fail(c, B200RT_ERR_NOT_DOMINANT, who + ": residual " + std::to_string(fin.true_res));
  return B200RT_OK;
}

}  // namespace

namespace api {

// Single-rank solves of different contexts on ONE device take turns: each is a cooperative launch that waits on its own
// barriers, and two such grids that each got part of the SMs would wait for each other's slots.  (Ranks of ONE solve that
// share a device -- the tests, a device group naming a device twice -- must run side by side and size their grids to fit.)
static std::mutex g_single_rank_solve[64];

int exchange_block(b200rt_ctx *c, void **dev_ptr) {
  if (!c->kry_xchg.p) {
    B200RT_CUDA(c, c->kry_xchg.ensure(sizeof(KryExchange)));
    B200RT_CUDA(c, cudaMemsetAsync(c->kry_xchg.p, 0, sizeof(KryExchange), c->stream));
    B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  if (dev_ptr) *dev_ptr = c->kry_xchg.p;
  return B200RT_OK;
}

int solve_distributed(b200rt_ctx *c, int rank, int world, void *const *blocks, bool reset_timer, int cta_cap) {
  // the systems: every singlet emission's (I - w K) S = S0 over the voxels, or the multiplet's (I - K) S = S0 over the
  // n_el = n_vox * n_upper elements (its branching is folded into K: multiplet_CFR_emission::pre_solve is empty)
  const bool mm = c->mult.defined;
  const int nu = mm ? c->mult.d.n_upper : 1;
  const int n = c->hg.n_vox * nu;
  if (world < 1 || world > KRY_MAX_WORLD || rank < 0 || rank >= world || !blocks)
    return fail(c, B200RT_ERR_ARG, "b200rt_solve_distributed: bad rank / world / blocks");
  if (n > KRY_MAX_N)
    return fail(c, B200RT_ERR_CAPACITY, "b200rt_solve_distributed: more than " + std::to_string(KRY_MAX_N) + " unknowns");
  struct System {
    bool have_K;
    const double *K, *S0;
    double *S;
    void *S_real;
    double branching;
    double *residual;
    bool *have_S, *rec_dirty;
  };
  std::vector<System> sys;
  if (mm) {
    Multiplet &M = c->mult;
    sys.push_back({M.have_K, M.K.as<double>(), M.S0.as<double>(), M.S.as<double>(), M.S_real.p, 1.0, &M.residual, &M.have_S,
                   &M.rec_dirty});
  } else {
    for (int e = 0; e < c->n_em; e++) {
      Emission &E = c->em[e];
      sys.push_back({E.have_K, E.K.as<double>(), E.S0.as<double>(), E.S.as<double>(), E.S_real.p, E.branching, &E.residual,
                     &E.have_S, &E.rec_dirty});
    }
  }
  if (int rc = exchange_block(c, nullptr)) return rc;
  if (blocks[rank] != c->kry_xchg.p)
    return fail(c, B200RT_ERR_ARG, "b200rt_solve_distributed: blocks[rank] is not this context's exchange block");
  if (reset_timer) PhaseTimer::reset(c);
  std::unique_lock<std::mutex> turn;
  if (world == 1) turn = std::unique_lock<std::mutex>(g_single_rank_solve[c->device & 63]);

  // the rows this rank multiplies: what its last influence call built (every element of each voxel)
  std::vector<int> rows;
  for (auto &r : c->built_ranges)
    for (int v = r.first; v < r.second; v++)
      for (int s = 0; s < nu; s++) rows.push_back(v * nu + s);
  KrySolver ks;
  if (int rc = kry_open(c, rows, n, nu, c->kry_work, c->kry_round_base, blocks, rank, world, cta_cap, 1, ks)) return rc;
  cudaStream_t s = c->stream;

  for (System &E : sys) {
    if (!E.have_K) return fail(c, B200RT_ERR_STATE, "b200rt_solve_distributed: influence rows not built");
    PhaseTimer t(c, PH_SOLVE);
    int launches = 0;
    B200RT_CUDA(c, kry_reset(ks, s));
    if (int rc = kry_setup(c, ks, E.K, E.branching, &launches)) return rc;
    bool fused = false;
    if (int rc = kry_iterate(c, ks, E.K, E.branching, E.S0, E.S, &launches, &fused)) return rc;
    B200RT_CUDA(c, cudaGetLastError());
    if (c->precision == B200RT_F64)
      B200RT_CUDA(c, launch_convert<double>(E.S, static_cast<double *>(E.S_real), n, s));
    else
      B200RT_CUDA(c, launch_convert<float>(E.S, static_cast<float *>(E.S_real), n, s));
    t.stop(launches);
    B200RT_CUDA(c, cudaMemcpyAsync(ks.h_st + 63, ks.wk.st, sizeof(KryState), cudaMemcpyDeviceToHost, s));
    B200RT_CUDA(c, cudaStreamSynchronize(s));
    const KryState fin = ks.h_st[63];
    kry_trace_report(ks, fused, fin);
    c->kry_round_base = fin.round;
    c->kry_last_iters = fin.iter;
    if (int rc = kry_status(c, fin, "b200rt_solve_distributed", " (rows missing on some rank, or a matrix the LU path should take)"))
      return rc;
    *E.residual = fin.true_res;
    *E.have_S = true;
    *E.rec_dirty = true;
  }
  PhaseTimer::collect(c);
  return B200RT_OK;
}

int solve_adjoint(b200rt_ctx *c, int e, int n_rhs, const double *rhs, double *lambda, int *n_steps, double *residual,
                  bool rows_complete) {
  const bool mm = c->mult.defined;
  if (mm ? e != 0 : (e < 0 || e >= c->n_em)) return fail(c, B200RT_ERR_ARG, "b200rt_solve_adjoint: bad emission index");
  if (n_rhs < 1 || !rhs || !lambda) return fail(c, B200RT_ERR_ARG, "b200rt_solve_adjoint: n_rhs < 1, or rhs / lambda NULL");
  const int nu = mm ? c->mult.d.n_upper : 1;
  const int n = c->hg.n_vox * nu;
  if (n > KRY_MAX_N)
    return fail(c, B200RT_ERR_CAPACITY, "b200rt_solve_adjoint: more than " + std::to_string(KRY_MAX_N) + " unknowns");
  if (!(mm ? c->mult.have_K : c->em[e].have_K)) return fail(c, B200RT_ERR_STATE, "b200rt_solve_adjoint: influence matrix not built");
  if (!rows_complete) {
    long long own = 0;
    for (auto &r : c->built_ranges) own += r.second - r.first;
    if (own != c->hg.n_vox)
      return fail(c, B200RT_ERR_STATE, "b200rt_solve_adjoint: this context did not build every row of K (a rank of a "
                                       "distributed job, or the solving rank of row sinks)");
  }
  const double *K = mm ? c->mult.K.as<double>() : c->em[e].K.as<double>();
  const double branching = mm ? 1.0 : c->em[e].branching;
  PhaseTimer::reset(c);
  // W^T w is zero when every weighted line of sight misses the grid: lambda = 0 without iterating
  std::vector<char> zero(n_rhs, 1);
  bool any = false;
  for (int k = 0; k < n_rhs; k++) {
    const double *r = rhs + (size_t) k * n;
    for (int i = 0; i < n && zero[k]; i++) zero[k] = r[i] == 0.0;
    any = any || !zero[k];
  }
  if (!any) {
    std::memset(lambda, 0, (size_t) n_rhs * n * sizeof(double));
    for (int k = 0; k < n_rhs; k++) {
      if (n_steps) n_steps[k] = 0;
      if (residual) residual[k] = 0.0;
    }
    return B200RT_OK;
  }

  std::unique_lock<std::mutex> turn(g_single_rank_solve[c->device & 63]);
  // its own exchange block and work area: the forward solve's round counters, which every rank of a distributed solve
  // must agree on, never see the adjoint's rounds
  if (!c->kry_adj_xchg.p) {
    B200RT_CUDA(c, c->kry_adj_xchg.ensure(sizeof(KryExchange)));
    B200RT_CUDA(c, cudaMemsetAsync(c->kry_adj_xchg.p, 0, sizeof(KryExchange), c->stream));
  }
  void *block = c->kry_adj_xchg.p;
  std::vector<int> rows(n);
  for (int i = 0; i < n; i++) rows[i] = i;
  KrySolver ks;
  if (int rc = kry_open(c, rows, n, nu, c->kry_adj_work, c->kry_adj_round_base, &block, 0, 1, 0, n_rhs, ks)) return rc;
  ks.trace = false;
  cudaStream_t s = c->stream;
  const size_t nb = (size_t) n_rhs * n * sizeof(double);
  B200RT_CUDA(c, c->kry_kt.ensure((size_t) n * n * sizeof(double)));
  B200RT_CUDA(c, c->kry_adj_io.ensure(2 * nb));
  double *d_rhs = c->kry_adj_io.as<double>(), *d_lam = d_rhs + (size_t) n_rhs * n;
  B200RT_CUDA(c, c->host_stage.ensure(nb));
  std::memcpy(c->host_stage.p, rhs, nb);
  B200RT_CUDA(c, cudaMemcpyAsync(d_rhs, c->host_stage.p, nb, cudaMemcpyHostToDevice, s));

  // K^T on every call: K can change under the context without its knowledge (row sinks, b200rt_influence_dev)
  {
    PhaseTimer t(c, PH_TRANSPOSE);
    const int tiles = (n + KT_TILE - 1) / KT_TILE;
    kry_transpose<<<dim3(tiles, tiles), dim3(KT_TILE, KT_ROWS), 0, s>>>(K, n, c->kry_kt.as<double>());
    B200RT_CUDA(c, cudaGetLastError());
    t.stop(1);
  }
  const double *Kt = c->kry_kt.as<double>();
  PhaseTimer t(c, PH_SOLVE);
  int launches = 0, last = -1;
  for (int k = 0; k < n_rhs; k++) {
    if (zero[k]) {
      B200RT_CUDA(c, cudaMemsetAsync(d_lam + (size_t) k * n, 0, (size_t) n * sizeof(double), s));
      continue;
    }
    B200RT_CUDA(c, kry_reset(ks, s));
    if (last < 0)
      if (int rc = kry_setup(c, ks, Kt, branching, &launches)) return rc;
    bool fused = false;
    if (int rc = kry_iterate(c, ks, Kt, branching, d_rhs + (size_t) k * n, d_lam + (size_t) k * n, &launches, &fused)) return rc;
    B200RT_CUDA(c, cudaMemcpyAsync(ks.h_st + 63 + k, ks.wk.st, sizeof(KryState), cudaMemcpyDeviceToHost, s));
    last = k;
  }
  B200RT_CUDA(c, cudaGetLastError());
  t.stop(launches);
  B200RT_CUDA(c, cudaMemcpyAsync(c->host_stage.p, d_lam, nb, cudaMemcpyDeviceToHost, s));
  B200RT_CUDA(c, cudaStreamSynchronize(s));
  c->kry_adj_round_base = ks.h_st[63 + last].round;
  for (int k = 0; k < n_rhs; k++) {
    if (zero[k]) {
      if (n_steps) n_steps[k] = 0;
      if (residual) residual[k] = 0.0;
      continue;
    }
    const KryState &fin = ks.h_st[63 + k];
    if (int rc = kry_status(c, fin, "b200rt_solve_adjoint (right-hand side " + std::to_string(k) + ")", "")) return rc;
    if (n_steps) n_steps[k] = fin.iter;
    if (residual) residual[k] = fin.true_res;
  }
  std::memcpy(lambda, c->host_stage.p, nb);
  PhaseTimer::collect(c);
  return B200RT_OK;
}

}  // namespace api
}  // namespace b200rt
