// influence.cu -- Holstein influence-matrix march and single scattering (sm_100a).
//
// Restates, for the device (reference src/):
//   singlet_CFR::update_tracker_start<true>        emission/singlet_CFR.hpp:80-260
//   singlet_CFR::update_tracker_influence          emission/singlet_CFR.hpp:352-370
//   singlet_CFR::compute_single_scattering         emission/singlet_CFR.hpp:372-398
//   singlet_CFR_tracker (lambda grid, weights)     emission/los_tracker.hpp:117-170
//   RT_grid::generate_S loop body                  RT_grid.hpp:166-201
//   emission_voxels::accumulate_influence          emission/emission_voxels.hpp:137-168
//
// It consumes the boundary lists written by traverse.cu, so no geometry is decided
// here; FMA contraction is allowed (results differ from the reference by rounding,
// ~1e-16 relative, against a 1e-6 tolerance).
//
// Mapping: a warp marches 8 rays at once, 4 lanes per ray, each lane carrying 5 of the
// 20 wavelength points (lambda index = sub + 4 m): the per-wavelength transmission
// vector P[] lives in registers, the per-step sum over wavelengths is two shuffles,
// and the step's contribution domega*G goes to K[row][voxel] with one fp64 RED.
//
// Per-voxel tables (march_table_kernel, once per emission) replace everything in the step that
// does not depend on the path length s:
//     kappa_i  = dtau_absorber + dtau_species * phi_i            (tau_i = kappa_i * s, as the reference rounds it)
//     wratio_i = w_i * dtau_species * phi_i / kappa_i
// so that  c_i = (1 - exp(-tau_i))/tau_i * (w_i phi_i P_i dtau_species s)  [singlet_CFR.hpp:141-159]
//              = wratio_i * P_i * (1 - exp(-tau_i))                        (s cancels: no division in the march)
// and, below the reference's series switch tau_i < 1e-3,  c_i = wratio_i * P_i * (1 - tau_i/2) * tau_i.
// The record of a voxel is laid out [lane 0..3][m 0..4]{kappa, wratio}: a lane reads its 80 bytes
// with five 16-byte loads, and the record of the NEXT step is fetched while the current one is
// integrated (software pipeline), because ncu showed the first version waiting on these loads.
// exp is fm::exp_nonpos in double (fastmath.cuh), expf in float.
#include "common.hpp"
#include "fastmath.cuh"

namespace b200rt {

namespace {

template <class Real> __device__ __forceinline__ Real rexp(Real x);
template <> __device__ __forceinline__ double rexp<double>(double x) { return exp(x); }
// exp(x), x <= 0.  GUARD: arguments may be astronomically negative (plane-parallel grid, fastmath.cuh)
template <class Real, bool GUARD> __device__ __forceinline__ Real exp_neg(Real x);
template <> __device__ __forceinline__ double exp_neg<double, false>(double x) { return fm::exp_nonpos(x); }
template <> __device__ __forceinline__ double exp_neg<double, true>(double x) { return fm::exp_nonpos_guarded(x); }
template <> __device__ __forceinline__ float exp_neg<float, false>(float x) { return expf(x); }
template <> __device__ __forceinline__ float exp_neg<float, true>(float x) { return expf(x); }
template <> __device__ __forceinline__ float rexp<float>(float x) { return expf(x); }
template <class Real> __device__ __forceinline__ Real rsqrt_(Real x);
template <> __device__ __forceinline__ double rsqrt_<double>(double x) { return sqrt(x); }
template <> __device__ __forceinline__ float rsqrt_<float>(float x) { return sqrtf(x); }

template <class Real>
__device__ __forceinline__ Real lambda2_of(int i) {
  // lambda(i) = i*delta_lambda, delta_lambda = lambda_max/(n_lambda-1)   (los_tracker.hpp:123-130)
  const Real delta_lambda = Real(4.0) / (N_LAMBDA - 1);
  Real l = i * delta_lambda;
  return l * l;
}
template <class Real>
__device__ __forceinline__ Real weight_of(int i) {
  const Real delta_lambda = Real(4.0) / (N_LAMBDA - 1);
  return (i == 0 || i == N_LAMBDA - 1) ? delta_lambda : Real(2.0) * delta_lambda;
}
template <class Real>
__device__ __forceinline__ Real one_over_sqrt_pi() { return (Real) 0.56418958354775628695; }

template <class Real>
__global__ void phi_table_kernel(const Real *__restrict__ T_ratio, int n_vox, Real *__restrict__ phi) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_vox * N_LAMBDA) return;
  const int v = idx / N_LAMBDA, i = idx % N_LAMBDA;
  phi[idx] = rexp<Real>(-lambda2_of<Real>(i) * T_ratio[v]);   // line_shape_function, los_tracker.hpp:142-147
}

constexpr int LANES_PER_RAY = 4;
constexpr int RAYS_PER_WARP = 32 / LANES_PER_RAY;
constexpr int LAMBDA_PER_LANE = N_LAMBDA / LANES_PER_RAY;   // 5
constexpr int MREC = 2 * N_LAMBDA;                          // Reals per voxel record

// march record of voxel v: [sub][m]{kappa, wratio}, lambda index i = sub + 4 m
template <class Real>
__global__ void march_table_kernel(const Real *__restrict__ phi, const Real *__restrict__ dts,
                                   const Real *__restrict__ dta, int n_vox, Real *__restrict__ mrec) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_vox * N_LAMBDA) return;
  const int v = idx / N_LAMBDA, i = idx % N_LAMBDA;
  const int sub = i % LANES_PER_RAY, m = i / LANES_PER_RAY;
  const Real ls = phi[idx];
  const Real kappa = dta[v] + dts[v] * ls;
  const Real wr = (kappa > 0) ? weight_of<Real>(i) * (dts[v] * ls) / kappa : Real(0);
  Real *o = mrec + (size_t) v * MREC + (sub * LAMBDA_PER_LANE + m) * 2;
  o[0] = kappa;
  o[1] = wr;
}

template <class Real> struct Rec2;      // {kappa, wratio} pair as one 16-byte (8-byte) load
template <> struct Rec2<double> { typedef double2 type; };
template <> struct Rec2<float> { typedef float2 type; };

// MODE 0: rows of the influence matrix (voxel-origin rays); MODE 1: sun-ward rays -> S0, tau
#ifndef MARCH_MIN_BLOCKS
#define MARCH_MIN_BLOCKS 2
#endif
template <class Real, int MODE, bool PP>
__global__ void __launch_bounds__(256, MARCH_MIN_BLOCKS)
march_kernel(GridView<Real> g, EmissionView<Real> em, int v_begin, long long n_rays_total,
             ListView<Real> lists, const int *__restrict__ shadow, double *__restrict__ K,
             double *__restrict__ S0, double *__restrict__ tau_sp_out, double *__restrict__ tau_abs_out,
             int *work_counter, unsigned long long *step_counter) {
  typedef typename Rec2<Real>::type R2;
  const int lane = threadIdx.x & 31;
  const int sub = lane & (LANES_PER_RAY - 1);
  const int grp = lane / LANES_PER_RAY;
  const int cap = lists.cap;
  const long long n_tasks = (n_rays_total + RAYS_PER_WARP - 1) / RAYS_PER_WARP;
  const R2 *__restrict__ mrec = reinterpret_cast<const R2 *>(em.mrec) + sub * LAMBDA_PER_LANE;

  Real w[LAMBDA_PER_LANE], l2[LAMBDA_PER_LANE];
#pragma unroll
  for (int m = 0; m < LAMBDA_PER_LANE; m++) {
    w[m] = weight_of<Real>(sub + LANES_PER_RAY * m);
    l2[m] = lambda2_of<Real>(sub + LANES_PER_RAY * m);
  }

  unsigned long long my_steps = 0;
  while (true) {
    long long task = 0;
    if (lane == 0) task = atomicAdd(work_counter, 1);
    task = __shfl_sync(0xffffffffu, task, 0);
    if (task >= n_tasks) break;

    const long long ray = task * RAYS_PER_WARP + grp;
    const bool valid = ray < n_rays_total;
    int len = 0, v0 = 0, ir = 0, mult = 1;
    if (valid) {
      len = lists.len[ray];
      if (MODE == 0) {
        v0 = v_begin + (int) (ray / g.n_rays);
        if (g.vox_map) v0 = g.vox_map[v0];
        ir = (int) (ray % g.n_rays);
        if (g.ray_mult) mult = g.ray_mult[ir];
      }
      else { v0 = (int) ray; if (shadow[v0]) len = -1; }
    }
    const Real Tr0 = valid ? em.T_ratio[v0] : Real(1);
    const Real renorm = one_over_sqrt_pi<Real>() * rsqrt_<Real>(Tr0);   // line_shape_normalization
    // P[m] carries norm(T0) * phi0_i * transmission_i: the line shape at the origin is constant along the ray, so it is
    // folded into the running product once instead of multiplying every step's contribution
    Real P[LAMBDA_PER_LANE];
#pragma unroll
    for (int m = 0; m < LAMBDA_PER_LANE; m++) P[m] = renorm * rexp<Real>(-l2[m] * Tr0);
    const Real domega = (MODE == 0 && valid) ? g.ray_domega[ir] : Real(1);   // march view: x the ray's multiplicity
    Real tau_sp = 0, tau_abs = 0;

    int maxlen = len;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) maxlen = max(maxlen, __shfl_xor_sync(0xffffffffu, maxlen, o));

    const Real *dl = lists.dist + (size_t) (valid ? ray : 0) * cap;
    const int *el = lists.ent + (size_t) (valid ? ray : 0) * cap;
    double *Krow = (MODE == 0) ? K + (size_t) v0 * g.n_vox : nullptr;

    // software pipeline: everything step k needs is loaded during step k-1
    Real d_prev = 0, d_cur = 0;
    int vox = 0, vox_next = 0;
    R2 rec[LAMBDA_PER_LANE];
#pragma unroll
    for (int m = 0; m < LAMBDA_PER_LANE; m++) rec[m] = R2{0, 0};
    if (len > 1) {
      d_prev = dl[0];
      d_cur = dl[1];
      vox = el[0];
      vox_next = el[1];
#pragma unroll
      for (int m = 0; m < LAMBDA_PER_LANE; m++) rec[m] = mrec[(size_t) vox * N_LAMBDA + m];
    }

    for (int k = 1; k < maxlen; k++) {
      const bool active = k < len;
      // ---- prefetch for step k+1
      const bool more = k + 1 < len;
      Real d_next = 0;
      int vox_next2 = 0;
      R2 rec_next[LAMBDA_PER_LANE];
      if (more) {
        d_next = dl[k + 1];
        vox_next2 = el[k + 1];
#ifdef B200RT_CHECKS
        if (vox_next < 0 || vox_next >= g.n_vox) printf("march<%d>: bad voxel %d ray=%lld k=%d len=%d\n", MODE, vox_next, ray, k, len);
#endif
#pragma unroll
        for (int m = 0; m < LAMBDA_PER_LANE; m++) rec_next[m] = mrec[(size_t) vox_next * N_LAMBDA + m];
      } else {
#pragma unroll
        for (int m = 0; m < LAMBDA_PER_LANE; m++) rec_next[m] = R2{0, 0};
      }
      // ---- step k: voxel `vox`, path length s
      Real G = 0;
      if (active) {
        const Real s = d_cur - d_prev;                                   // boundaries.hpp:366,376
        if (MODE == 1) { tau_sp += em.dtau_species[vox] * s; tau_abs += em.dtau_absorber[vox] * s; }
#pragma unroll
        for (int m = 0; m < LAMBDA_PER_LANE; m++) {
          const Real tau = rec[m].x * s;
          const Real tp = exp_neg<Real, PP>(-tau);
          if (MODE == 0) {
            const Real f = ((double) tau < 1e-3) ? (Real(1.0) - Real(0.5) * tau) * tau : (Real(1.0) - tp);
            G = fma(rec[m].y * P[m], f, G);
          }
          P[m] *= tp;
        }
      }
      if (MODE == 0) {
        G += __shfl_xor_sync(0xffffffffu, G, 1);
        G += __shfl_xor_sync(0xffffffffu, G, 2);
        if (active && sub == 0) atomicAdd(&Krow[vox], (double) (domega * G));
      }
      d_prev = d_cur; d_cur = d_next;
      vox = vox_next; vox_next = vox_next2;
#pragma unroll
      for (int m = 0; m < LAMBDA_PER_LANE; m++) rec[m] = rec_next[m];
    }
    if (MODE == 0) {
      if (sub == 0 && len > 1) my_steps += (unsigned long long) (len - 1) * mult;   // the reference's count
    } else {
      // holstein_T_final = sum_i w_i * norm(T0) * phi0_i * P_i   (singlet_CFR.hpp:183-186)
      Real T = 0;
#pragma unroll
      for (int m = 0; m < LAMBDA_PER_LANE; m++) T += w[m] * P[m];
      T += __shfl_xor_sync(0xffffffffu, T, 1);
      T += __shfl_xor_sync(0xffffffffu, T, 2);
      if (valid && sub == 0) {
        if (len == -1) { S0[v0] = 0.0; tau_sp_out[v0] = -1.0; tau_abs_out[v0] = -1.0; }   // behind the limb
        else if (len <= 1) { S0[v0] = 1.0; tau_sp_out[v0] = 0.0; tau_abs_out[v0] = 0.0; } // tracker reset values
        else { S0[v0] = (double) T; tau_sp_out[v0] = (double) tau_sp; tau_abs_out[v0] = (double) tau_abs; }
      }
    }
  }
  if (MODE == 0 && step_counter) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) my_steps += __shfl_xor_sync(0xffffffffu, my_steps, o);
    if (lane == 0 && my_steps) atomicAdd(step_counter, my_steps);
  }
}

} // namespace

template <class Real>
cudaError_t launch_phi_table(const Real *T_ratio, const Real *dts, const Real *dta, int n_vox, Real *phi, Real *mrec,
                             cudaStream_t s) {
  const int n = n_vox * N_LAMBDA;
  phi_table_kernel<Real><<<(n + 255) / 256, 256, 0, s>>>(T_ratio, n_vox, phi);
  march_table_kernel<Real><<<(n + 255) / 256, 256, 0, s>>>(phi, dts, dta, n_vox, mrec);
  return cudaGetLastError();
}

template <class Real>
cudaError_t launch_influence(const GridView<Real> &g, const EmissionView<Real> &em, int v_begin, int v_end,
                             ListView<Real> lists, double *K, int *work_counter,
                             unsigned long long *step_counter, cudaStream_t s) {
  const long long n = (long long) (v_end - v_begin) * g.n_rays;
  if (n <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), s);
  if (e != cudaSuccess) return e;
  const int threads = 256;
  const long long tasks = (n + RAYS_PER_WARP - 1) / RAYS_PER_WARP;
  long long blocks = (tasks + threads / 32 - 1) / (threads / 32);
  const long long persistent = (long long) NUM_SMS * 4;
  if (blocks > persistent) blocks = persistent;
  if (g.pp)
    march_kernel<Real, 0, true><<<(unsigned) blocks, threads, 0, s>>>(g, em, v_begin, n, lists, nullptr, K, nullptr, nullptr,
                                                                      nullptr, work_counter, step_counter);
  else
    march_kernel<Real, 0, false><<<(unsigned) blocks, threads, 0, s>>>(g, em, v_begin, n, lists, nullptr, K, nullptr, nullptr,
                                                                       nullptr, work_counter, step_counter);
  return cudaGetLastError();
}

template <class Real>
cudaError_t launch_single_scattering(const GridView<Real> &g, const EmissionView<Real> &em, ListView<Real> lists,
                                     const int *shadow, double *S0, double *tau_sp, double *tau_abs,
                                     int *work_counter, cudaStream_t s) {
  const long long n = g.n_vox;
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), s);
  if (e != cudaSuccess) return e;
  const int threads = 256;
  const long long tasks = (n + RAYS_PER_WARP - 1) / RAYS_PER_WARP;
  long long blocks = (tasks + threads / 32 - 1) / (threads / 32);
  if (blocks > NUM_SMS * 4) blocks = NUM_SMS * 4;
  if (g.pp)
    march_kernel<Real, 1, true><<<(unsigned) blocks, threads, 0, s>>>(g, em, 0, n, lists, shadow, nullptr, S0, tau_sp, tau_abs,
                                                                      work_counter, nullptr);
  else
    march_kernel<Real, 1, false><<<(unsigned) blocks, threads, 0, s>>>(g, em, 0, n, lists, shadow, nullptr, S0, tau_sp, tau_abs,
                                                                       work_counter, nullptr);
  return cudaGetLastError();
}

template cudaError_t launch_phi_table<double>(const double *, const double *, const double *, int, double *, double *, cudaStream_t);
template cudaError_t launch_phi_table<float>(const float *, const float *, const float *, int, float *, float *, cudaStream_t);
template cudaError_t launch_influence<double>(const GridView<double> &, const EmissionView<double> &, int, int,
                                              ListView<double>, double *, int *, unsigned long long *, cudaStream_t);
template cudaError_t launch_influence<float>(const GridView<float> &, const EmissionView<float> &, int, int,
                                             ListView<float>, double *, int *, unsigned long long *, cudaStream_t);
template cudaError_t launch_single_scattering<double>(const GridView<double> &, const EmissionView<double> &,
                                                      ListView<double>, const int *, double *, double *, double *,
                                                      int *, cudaStream_t);
template cudaError_t launch_single_scattering<float>(const GridView<float> &, const EmissionView<float> &,
                                                     ListView<float>, const int *, double *, double *, double *,
                                                     int *, cudaStream_t);

} // namespace b200rt
