// los_march.cuh -- the per-sub-step pieces of the singlet line-of-sight march that the brightness kernel (brightness.cu)
// and the line-of-sight weighting functions (los_weights.cu) share: the 4-lane group layout, the interleaved voxel
// records and their 4-corner interpolation, and the line shapes of one sub-step.
#pragma once
#include "common.hpp"
#include "fastmath.cuh"
#include "los_geom.cuh"

namespace b200rt {

namespace {

constexpr int LPR = 4;                       // lanes per line of sight
constexpr int NLL = N_LAMBDA / LPR;          // wavelength points per lane (5)
constexpr int REC = 8;                       // Reals per voxel record: T_ratio, density, dtau_species, dtau_absorber, S, pad

template <class Real>
__device__ __forceinline__ Real shfl_real(unsigned mask, Real v, int src) { return __shfl_sync(mask, v, src); }

// 4-corner interpolation of one voxel record: s = sum_k w[k]*q[idx[k]] left to right
// (emission_voxels.hpp:58-70) for the five quantities at once
template <class Real>
__device__ __forceinline__ void interp_record(const Real *__restrict__ tab, const int (&idx)[4], const Real (&w)[4],
                                              Real (&o)[5]);
template <>
__device__ __forceinline__ void interp_record<double>(const double *__restrict__ tab, const int (&idx)[4],
                                                      const double (&w)[4], double (&o)[5]) {
#pragma unroll
  for (int q = 0; q < 5; q++) o[q] = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const double2 *p = reinterpret_cast<const double2 *>(tab + (size_t) idx[k] * REC);
    const double2 a = __ldg(p), b = __ldg(p + 1);
    const double c = __ldg(tab + (size_t) idx[k] * REC + 4);
    o[0] += w[k] * a.x; o[1] += w[k] * a.y; o[2] += w[k] * b.x; o[3] += w[k] * b.y; o[4] += w[k] * c;
  }
}
template <>
__device__ __forceinline__ void interp_record<float>(const float *__restrict__ tab, const int (&idx)[4],
                                                     const float (&w)[4], float (&o)[5]) {
#pragma unroll
  for (int q = 0; q < 5; q++) o[q] = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const float4 a = __ldg(reinterpret_cast<const float4 *>(tab + (size_t) idx[k] * REC));
    const float c = __ldg(tab + (size_t) idx[k] * REC + 4);
    o[0] += w[k] * a.x; o[1] += w[k] * a.y; o[2] += w[k] * a.z; o[3] += w[k] * a.w; o[4] += w[k] * c;
  }
}

// per-lane line shapes of one sub-step.  double: from q = exp(-dl^2 T) by products; float: expf
template <class Real> struct LineShape;
template <> struct LineShape<double> {
  // what the geometry lane broadcasts
  __device__ static double param(double Tr) {
    const double dl = 4.0 / (N_LAMBDA - 1);
    return fm::exp_nonpos(-(dl * dl) * Tr);
  }
  __device__ static void eval(double q, int sub, double (&phi)[NLL]) {
    const double q2 = q * q, q4 = q2 * q2, q8 = q4 * q4, q16 = q8 * q8, q32 = q16 * q16;
    // phi_sub = q^(sub^2); D = q^(8 sub + 16); phi_{i+4} = phi_i * D; D *= q^32
    double p = (sub == 0) ? 1.0 : (sub == 1) ? q : (sub == 2) ? q4 : q8 * q;
    double D = (sub == 0) ? q16 : (sub == 1) ? q16 * q8 : (sub == 2) ? q32 : q32 * q8;
#pragma unroll
    for (int m = 0; m < NLL; m++) {
      phi[m] = p;
      p *= D;
      D *= q32;
    }
  }
};
template <> struct LineShape<float> {
  // the same products in float: phi_i = q^(i^2) carries ~i^2 x 6e-8 relative error, weighted by phi_i itself in the sum
  // (1e-6 on the line integral against the 1e-4 bar); one expf per sub-step instead of five per lane
  __device__ static float param(float Tr) {
    const float dl = 4.0f / (N_LAMBDA - 1);
    return expf(-(dl * dl) * Tr);
  }
  __device__ static void eval(float q, int sub, float (&phi)[NLL]) {
    const float q2 = q * q, q4 = q2 * q2, q8 = q4 * q4, q16 = q8 * q8, q32 = q16 * q16;
    float p = (sub == 0) ? 1.0f : (sub == 1) ? q : (sub == 2) ? q4 : q8 * q;
    float D = (sub == 0) ? q16 : (sub == 1) ? q16 * q8 : (sub == 2) ? q32 : q32 * q8;
#pragma unroll
    for (int m = 0; m < NLL; m++) {
      phi[m] = p;
      p *= D;
      D *= q32;
    }
  }
};

} // namespace

} // namespace b200rt
