// multiplet.cu -- multiplet CFR emissions on the device (sm_100a): influence matrix, single scattering,
// line-of-sight brightness for O I 102.6 nm, the H Lyman alpha/beta fine-structure multiplet and the
// singlet-through-the-multiplet-code check.
//
// Restates, for the device (reference src/):
//   multiplet_CFR_emission::update_tracker_start<influence>      emission/multiplet_CFR_emission.hpp:69-300
//   multiplet_CFR_emission::update_tracker_influence             emission/multiplet_CFR_emission.hpp:382-404
//   multiplet_CFR_emission::update_tracker_brightness            emission/multiplet_CFR_emission.hpp:302-316
//   multiplet_CFR_emission::update_tracker_start_interp          emission/multiplet_CFR_emission.hpp:352-378
//   O_1026_emission / H_lyman_multiplet::compute_single_scattering   emission/O_1026.hpp:84-131, H_lyman_multiplet.hpp:118-157
//   O_1026_tracker / H_lyman_multiplet_tracker / H_lyman_singlet_tracker (line shapes, weights, reset, exits_bottom)
//                                                                 emission/O_1026_tracker.hpp:199-291, H_multiplet_tracker*.hpp
//   emission_voxels (element order voxel*n_upper+state, accumulate_influence, brightness interp)
//                                                                 emission/emission_voxels.hpp:32, 58-70, 137-155, 199-233
//
// Mapping.  A ray (or line of sight) belongs to a group of 8 lanes; lane `sub` carries the wavelength points
// i = sub + 8 j (j < NLP = ceil(n_lambda / 8)) of EVERY multiplet, so the transmission vectors P[m][.] stay in
// registers and the per-step sums over wavelength are three shuffle stages.  Four rays per warp.
//
// Influence march.  Everything of a step that does not depend on the path length s is tabulated per voxel once per
// emission (mult_table_kernel):
//     kappa[m][i]   = sum over member lines ( n_lower sigma ls(line,i,T) + n_abs xsec(line) )        (:98-117; the absorber
//                     term is added once PER MEMBER LINE, which the reference does and parity requires)
//     wlsk[line][i] = weight(line) ls(line,i,T) / kappa[mult(line)][i]
// so that the reference's  (1-exp(-tau))/tau * weight ls P s  (:168-196) is  wlsk * P * (1 - exp(-tau)): the path length
// cancels and the march has no division (below the series switch tau < 1e-3: wlsk P (1 - tau/2) tau).  The origin voxel
// contributes c0[line][i] = sigma(line) n0_lower / decay(upper) * ls(line,i,T0) (:245-279), held in registers per ray.
// G[iu][ju] is reduced over the group and lands in K[(v0,iu),(v,ju)] with fp64 REDs (K stays resident in HBM).
//
// The index tables (which line belongs to which multiplet / lower / upper state) are compile-time traits so that every
// register array is indexed by constants after unrolling; the numeric line parameters arrive by value (MultParams).
#include "common.hpp"
#include "fastmath.cuh"
#include "los_geom.cuh"

namespace b200rt {

namespace {

struct TraitsO {   // O_1026_constants_detail, O_1026_tracker.hpp:11-24,188
  static constexpr int KIND = B200RT_MULT_O1026, NL = 6, NM = 3, NLOW = 3, NUP = 3, NLAM = 21;
  __host__ __device__ static constexpr int mult(int l) { return l == 0 ? 0 : (l < 3 ? 1 : 2); }
  __host__ __device__ static constexpr int lower(int l) { return l == 0 ? 0 : (l < 3 ? 1 : 2); }
  __host__ __device__ static constexpr int upper(int l) { return l == 0 ? 0 : l == 1 ? 0 : l == 2 ? 1 : l == 3 ? 0 : l == 4 ? 1 : 2; }
};
struct TraitsH {   // H_lyman_multiplet_constants_detail, H_multiplet_tracker.hpp:11-20,146
  static constexpr int KIND = B200RT_MULT_H_LYMAN, NL = 4, NM = 2, NLOW = 1, NUP = 4, NLAM = 41;
  __host__ __device__ static constexpr int mult(int l) { return l < 2 ? 0 : 1; }
  __host__ __device__ static constexpr int lower(int) { return 0; }
  __host__ __device__ static constexpr int upper(int l) { return l; }
};
struct TraitsS {   // H_lyman_singlet_constants_detail, H_multiplet_tracker_test.hpp:11-20
  static constexpr int KIND = B200RT_MULT_H_SINGLET, NL = 2, NM = 2, NLOW = 1, NUP = 2, NLAM = 41;
  __host__ __device__ static constexpr int mult(int l) { return l; }
  __host__ __device__ static constexpr int lower(int) { return 0; }
  __host__ __device__ static constexpr int upper(int l) { return l; }
};

constexpr int LPR = MULT_LPR;
constexpr int RPW = 32 / LPR;   // rays per warp
template <class TR> struct Dim {
  static constexpr int NLP = (TR::NLAM + LPR - 1) / LPR;   // wavelength points per lane
  static constexpr int RS = TR::NM + TR::NL;               // Reals per wavelength point in the step record
};

template <class Real> __device__ __forceinline__ Real m_exp(Real x);          // x <= 0
template <> __device__ __forceinline__ double m_exp<double>(double x) { return fm::exp_nonpos_guarded(x); }   // also on plane-parallel grids
template <> __device__ __forceinline__ float m_exp<float>(float x) { return expf(x); }
template <class Real> __device__ __forceinline__ Real m_sqrt(Real x);
template <> __device__ __forceinline__ double m_sqrt<double>(double x) { return sqrt(x); }
template <> __device__ __forceinline__ float m_sqrt<float>(float x) { return (float) sqrt((double) x); }   // unqualified sqrt: double

template <class Real>
__device__ __forceinline__ Real group_sum(Real v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  return v;
}

// ---------------------------------------------------------------- per-voxel tables
template <class Real, class TR>
__global__ void mult_table_kernel(MultView<Real> mv, MultParams<Real> P, int n_vox) {
  constexpr int NL = TR::NL, NM = TR::NM, NLP = Dim<TR>::NLP, RS = Dim<TR>::RS;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_vox * LPR * NLP) return;
  const int v = idx / (LPR * NLP), i = idx % (LPR * NLP);
  const int lane = i % LPR, j = i / LPR;
  Real *rs = mv.rec_step + ((size_t) (v * LPR + lane) * NLP + j) * RS;
  Real *ro = mv.rec_org + ((size_t) (v * LPR + lane) * NLP + j) * NL;
  Real *rw = mv.rec_w0 + ((size_t) (v * LPR + lane) * NLP + j) * NL;
  if (i >= TR::NLAM) {   // padding wavelength slots: no opacity, no weight
#pragma unroll
    for (int q = 0; q < RS; q++) rs[q] = 0;
#pragma unroll
    for (int l = 0; l < NL; l++) { ro[l] = 0; rw[l] = 0; }
    return;
  }
  const Real T = mv.T[v], nabs = mv.nabs[v];
  const Real a = P.T_ref / T;
  const Real nf = m_sqrt<Real>(a);
  const Real lam = -P.lambda_max + i * P.delta_lambda;
  Real ls[NL], kappa[NM];
#pragma unroll
  for (int m = 0; m < NM; m++) kappa[m] = 0;
#pragma unroll
  for (int l = 0; l < NL; l++) {
    const Real x = lam - P.offset[l];
    const Real nrm = P.norm[l] * nf;
    ls[l] = nrm * m_exp<Real>(-(x * x) * a);
    const Real nl = mv.n[TR::lower(l)][v];
    kappa[TR::mult(l)] += nl * P.sigma[l] * ls[l] + nabs * P.xsec[l];
    ro[l] = P.sigma[l] * nl / P.decay[TR::upper(l)] * ls[l];
    rw[l] = P.weight[l] * ls[l];
    if (i == 0) {
      mv.tsv[(size_t) v * NL + l] = nl * P.sigma[l] * nrm;
      mv.tav[(size_t) v * NL + l] = nabs * P.xsec[l];
    }
  }
#pragma unroll
  for (int m = 0; m < NM; m++) rs[m] = kappa[m];
#pragma unroll
  for (int l = 0; l < NL; l++) {
    const Real k = kappa[TR::mult(l)];
    rs[NM + l] = (k > 0) ? P.weight[l] * ls[l] / k : Real(0);
  }
}

// brightness records: {T, n_abs, n[NLOW], S[NUP]} of the voxel points (interpolated) and of the voxel averages (nointerp)
template <class Real, class TR>
__global__ void mult_pack_kernel(MultView<Real> mv, int n_vox) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_vox) return;
  Real *p = mv.rec_pt + (size_t) v * MULT_REC, *a = mv.rec_avg + (size_t) v * MULT_REC;
#pragma unroll
  for (int q = 0; q < MULT_REC; q++) { p[q] = 0; a[q] = 0; }
  p[0] = mv.T_pt[v]; p[1] = mv.nabs_pt[v];
  a[0] = mv.T[v]; a[1] = mv.nabs[v];
#pragma unroll
  for (int l = 0; l < TR::NLOW; l++) { p[2 + l] = mv.n_pt[l][v]; a[2 + l] = mv.n[l][v]; }
#pragma unroll
  for (int u = 0; u < TR::NUP; u++) { p[5 + u] = mv.S[(size_t) v * TR::NUP + u]; a[5 + u] = mv.S[(size_t) v * TR::NUP + u]; }
}

// ---------------------------------------------------------------- influence march / single scattering
// MODE 0: voxel-origin rays -> rows of K;  MODE 1: sun-ward rays -> singlescat, single-scattering optical depths
template <class Real, class TR, int MODE>
__global__ void __launch_bounds__(128)
mult_march_kernel(GridView<Real> g, MultView<Real> mv, MultParams<Real> P_, int v_begin, long long n_rays_total,
                  ListView<Real> lists, const int *__restrict__ shadow, double *__restrict__ K,
                  double *__restrict__ S0, double *__restrict__ tsp_out, double *__restrict__ tab_out,
                  int *work_counter, unsigned long long *step_counter) {
  constexpr int NL = TR::NL, NM = TR::NM, NUP = TR::NUP, NLP = Dim<TR>::NLP, RS = Dim<TR>::RS;
  const int lane = threadIdx.x & 31;
  const int sub = lane & (LPR - 1);
  const int grp = lane / LPR;
  const int cap = lists.cap;
  const long long n_tasks = (n_rays_total + RPW - 1) / RPW;
  const size_t NE = (size_t) g.n_vox * NUP;

  unsigned long long my_steps = 0;
  while (true) {
    long long task = 0;
    if (lane == 0) task = atomicAdd(work_counter, 1);
    task = __shfl_sync(0xffffffffu, task, 0);
    if (task >= n_tasks) break;

    const long long ray = task * RPW + grp;
    const bool valid = ray < n_rays_total;
    int len = 0, v0 = 0, ir = 0, mult = 1;
    if (valid) {
      len = lists.len[ray];
      if (MODE == 0) {
        v0 = v_begin + (int) (ray / g.n_rays);
        if (g.vox_map) v0 = g.vox_map[v0];       // interleaved shards: local slot -> source voxel
        ir = (int) (ray % g.n_rays);
        if (g.ray_mult) mult = g.ray_mult[ir];
      }
      else { v0 = (int) ray; if (shadow[v0]) len = -1; }
    }
    // origin factors: c0 (MODE 0) or weight*ls0 (MODE 1)
    Real org[NL][NLP];
    {
      const Real *ro = (MODE == 0 ? mv.rec_org : mv.rec_w0) + ((size_t) (v0 * LPR + sub) * NLP) * NL;
#pragma unroll
      for (int j = 0; j < NLP; j++)
#pragma unroll
        for (int l = 0; l < NL; l++) org[l][j] = valid ? ro[j * NL + l] : Real(0);
    }
    Real P[NM][NLP];
#pragma unroll
    for (int m = 0; m < NM; m++)
#pragma unroll
      for (int j = 0; j < NLP; j++) P[m][j] = Real(1);
    const Real domega = (MODE == 0 && valid) ? g.ray_domega[ir] : Real(1);   // march view: x the ray's multiplicity
    Real tsp[NL], tab[NL];
#pragma unroll
    for (int l = 0; l < NL; l++) { tsp[l] = 0; tab[l] = 0; }

    int maxlen = len;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) maxlen = max(maxlen, __shfl_xor_sync(0xffffffffu, maxlen, o));
    const Real *dl = lists.dist + (size_t) (valid ? ray : 0) * cap;
    const int *el = lists.ent + (size_t) (valid ? ray : 0) * cap;

    for (int k = 1; k < maxlen; k++) {
      const bool active = k < len;
      Real G[NUP][NUP];
#pragma unroll
      for (int a = 0; a < NUP; a++)
#pragma unroll
        for (int b = 0; b < NUP; b++) G[a][b] = 0;
      int vox = 0;
      if (active) {
        vox = el[k - 1];
        const Real s = dl[k] - dl[k - 1];                      // boundaries.hpp:366,376
        const Real *r = mv.rec_step + ((size_t) (vox * LPR + sub) * NLP) * RS;
        if (MODE == 1) {
#pragma unroll
          for (int l = 0; l < NL; l++) { tsp[l] += mv.tsv[(size_t) vox * NL + l] * s; tab[l] += mv.tav[(size_t) vox * NL + l] * s; }
        }
#pragma unroll
        for (int j = 0; j < NLP; j++) {
          Real base[NM];
#pragma unroll
          for (int m = 0; m < NM; m++) {
            const Real tau = r[j * RS + m] * s;
            const Real p = m_exp<Real>(-tau);
            const Real f = ((double) tau < 1e-3) ? (Real(1.0) - Real(0.5) * tau) * tau : (Real(1.0) - p);
            base[m] = f * P[m][j];
            P[m][j] *= p;
          }
          if (MODE == 0) {
            Real cA[NL];
#pragma unroll
            for (int lc = 0; lc < NL; lc++) cA[lc] = base[TR::mult(lc)] * r[j * RS + NM + lc] * P_.A[lc];
#pragma unroll
            for (int lo = 0; lo < NL; lo++)
#pragma unroll
              for (int lc = 0; lc < NL; lc++)
                if (TR::mult(lo) == TR::mult(lc)) G[TR::upper(lo)][TR::upper(lc)] += org[lo][j] * cA[lc];
          }
        }
      }
      if (MODE == 0) {
        double *Kbase = K + ((size_t) v0 * NUP) * NE + (size_t) vox * NUP;
#pragma unroll
        for (int a = 0; a < NUP; a++)
#pragma unroll
          for (int b = 0; b < NUP; b++) {
            const Real gsum = group_sum<Real>(G[a][b]);
            if (active && sub == ((a * NUP + b) & (LPR - 1)) && gsum != 0) atomicAdd(Kbase + (size_t) a * NE + b, (double) (domega * gsum));
          }
      }
    }
    if (MODE == 0) {
      if (sub == 0 && len > 1) my_steps += (unsigned long long) (len - 1) * mult;   // the reference's count
    } else {
      // holstein_T_final[line] = sum_i weight ls0 P_final   (multiplet_CFR_emission.hpp:222-228)
#pragma unroll
      for (int l = 0; l < NL; l++) {
        Real T = 0;
#pragma unroll
        for (int j = 0; j < NLP; j++) T += org[l][j] * P[TR::mult(l)][j];
        T = group_sum<Real>(T);
        if (valid && sub == 0) {
          const bool dark = (len == -1);
          tsp_out[(size_t) v0 * NL + l] = dark ? -1.0 : (double) tsp[l];
          tab_out[(size_t) v0 * NL + l] = dark ? -1.0 : (double) tab[l];
          if (P_.pumped[l]) {
            const Real exc = P_.solar[l] * mv.n[TR::lower(l)][v0] * P_.sigma[l] / P_.decay[TR::upper(l)];
            S0[(size_t) v0 * NUP + TR::upper(l)] = dark ? 0.0 : (double) (exc * T);
          }
        }
      }
    }
  }
  if (MODE == 0 && step_counter) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) my_steps += __shfl_xor_sync(0xffffffffu, my_steps, o);
    if (lane == 0 && my_steps) atomicAdd(step_counter, my_steps);
  }
}

// ---------------------------------------------------------------- brightness
// RT_grid::brightness (RT_grid.hpp:233-299): 8 lanes per line of sight; lane q does the geometry of sub-step j0+q
// (extend, interp_weights, 4-corner gathers of one record per voxel), then the 8 sub-steps are applied in order.
template <class Real, class TR>
__global__ void __launch_bounds__(128)
mult_brightness_kernel(GridView<Real> g, MultView<Real> mv, MultParams<Real> P_, const Real *__restrict__ los_in,
                       long long los_stride, long long first, long long count, ListView<Real> lists, int n_subsamples,
                       Real *__restrict__ out, long long n_los_total, int *queue, const int *__restrict__ order) {
  constexpr int NL = TR::NL, NM = TR::NM, NLOW = TR::NLOW, NUP = TR::NUP, NLP = Dim<TR>::NLP;
  constexpr int NQ = 2 + NLOW + NUP;     // record entries in use
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n_rb = g.n_rb, n_sb = g.n_sb, n_sb1 = n_sb - 1;
  GeomTables<Real> T;
  T.load(smem_raw, g);

  const int lane = threadIdx.x & 31;
  const int sub = lane & (LPR - 1);
  const int lead = lane & ~(LPR - 1);
  const unsigned gmask = 0xFFu << lead;
  const bool interp = n_subsamples != 0;
  const int nsd = interp ? n_subsamples : 2;
  const int nss = nsd - 1;
  const Real eps = MathB<Real>::eps();
  const Real scale = Real(1e9);
  const Real r_scale = MathB<Real>::rcp_(scale), r_nss = MathB<Real>::rcp_((Real) (nsd - 1));

  bool have = false, exhausted = false;
  long long los = 0;
  int total = 0, j0 = 0, flagbits = 0;
  const Real *dl = nullptr;
  const int *el = nullptr;
  Real px = 0, py = 0, pz = 0, lx = 0, ly = 0, lz = 0;
  Real P[NM][NLP], accB[NL], acc_tsp[NL], acc_tab[NL], acc_col[NLOW];
  const size_t n_out = 3 * NL + NLOW;

  while (true) {
    while (!have && !exhausted) {
      int t = 0;
      if (sub == 0) t = atomicAdd(queue, 1);
      t = __shfl_sync(gmask, t, lead);
      if (t >= count) { exhausted = true; break; }
      if (order) t = order[t];      // longest lines of sight first (launch_los_order, brightness.cu)
      los = first + t;
      const int len = lists.len[t];
      if (len <= 0) {     // misses the grid: tracker reset values
        for (int q = sub; q < (int) n_out; q += LPR) out[(size_t) q * n_los_total + los] = Real(0);
        continue;
      }
      total = (len - 1) * nss;
      flagbits = lists.flag[t];
      dl = lists.dist + (size_t) t * lists.cap;
      el = lists.ent + (size_t) t * lists.cap;
      px = MathB<Real>::divc_(los_in[0 * los_stride + los], scale, r_scale);
      py = MathB<Real>::divc_(los_in[1 * los_stride + los], scale, r_scale);
      pz = MathB<Real>::divc_(los_in[2 * los_stride + los], scale, r_scale);
      lx = los_in[5 * los_stride + los]; ly = los_in[6 * los_stride + los]; lz = los_in[7 * los_stride + los];
#pragma unroll
      for (int l = 0; l < NL; l++) { accB[l] = 0; acc_tsp[l] = 0; acc_tab[l] = 0; }
#pragma unroll
      for (int l = 0; l < NLOW; l++) acc_col[l] = 0;
#pragma unroll
      for (int m = 0; m < NM; m++)
#pragma unroll
        for (int j = 0; j < NLP; j++) P[m][j] = Real(1);
      j0 = 0;
      have = true;
    }
    if (__all_sync(0xffffffffu, !have)) break;

    // ---- geometry of sub-step j0+sub
    Real my_s = 0;
    Real my_in[NQ];
#pragma unroll
    for (int q = 0; q < NQ; q++) my_in[q] = 0;
    const int jj = j0 + sub;
    if (have && jj < total) {
      const int ib = jj / nss + 1;
      const int is = jj - (ib - 1) * nss + 1;
      Real d_start = dl[ib - 1];
      const Real dnext = dl[ib];
      const int cur = el[ib - 1];
      Real d_step = MathB<Real>::divc_(dnext - d_start, (Real) (nsd - 1), r_nss);
      d_start += Real(0.5) * eps * d_step;          // RT_grid.hpp:268-271
      d_step *= Real(1.0) - eps;
      my_s = d_step;
      if (!interp) {
        const Real *r = mv.rec_avg + (size_t) cur * MULT_REC;
        my_in[0] = r[0]; my_in[1] = r[1];
#pragma unroll
        for (int l = 0; l < NLOW; l++) my_in[2 + l] = r[2 + l];
#pragma unroll
        for (int u = 0; u < NUP; u++) my_in[2 + NLOW + u] = r[5 + u];
      } else {
        int idx[4];
        Real w[4];
        const Real dist = d_start + is * d_step;
        substep_interp<Real>(T, cur, px, py, pz, lx, ly, lz, dist, idx, w);
#pragma unroll
        for (int k = 0; k < 4; k++) {              // interp_voxel_vector: sum_k w[k] * q[idx[k]], left to right
          const Real *r = mv.rec_pt + (size_t) idx[k] * MULT_REC;
          my_in[0] += w[k] * r[0]; my_in[1] += w[k] * r[1];
#pragma unroll
          for (int l = 0; l < NLOW; l++) my_in[2 + l] += w[k] * r[2 + l];
#pragma unroll
          for (int u = 0; u < NUP; u++) my_in[2 + NLOW + u] += w[k] * r[5 + u];
        }
      }
    }

    // ---- apply the eight sub-steps in order
    const int nvalid = have ? min(LPR, total - j0) : 0;
    // (broadcasts and wavelength sums as full-warp shuffles executed by every lane: see brightness.cu)
    const unsigned FULL = 0xffffffffu;
    for (int q = 0; q < LPR; q++) {
      {
        const bool act = q < nvalid;
        const Real s = __shfl_sync(FULL, my_s, lead + q);
        Real in[NQ];
#pragma unroll
        for (int a = 0; a < NQ; a++) in[a] = __shfl_sync(FULL, my_in[a], lead + q);
        const Real T = act ? in[0] : Real(1), nabs = in[1];
        const Real a = P_.T_ref / T;
        const Real nf = m_sqrt<Real>(a);
        Real Tint[NL];
#pragma unroll
        for (int l = 0; l < NL; l++) Tint[l] = 0;
        if (act)
#pragma unroll
        for (int j = 0; j < NLP; j++) {
          const int i = sub + LPR * j;
          const Real lam = -P_.lambda_max + i * P_.delta_lambda;
          const bool ok = i < TR::NLAM;
          Real ls[NL], kap[NM];
#pragma unroll
          for (int m = 0; m < NM; m++) kap[m] = 0;
#pragma unroll
          for (int l = 0; l < NL; l++) {
            const Real x = lam - P_.offset[l];
            ls[l] = (P_.norm[l] * nf) * m_exp<Real>(-(x * x) * a);
            kap[TR::mult(l)] += in[2 + TR::lower(l)] * P_.sigma[l] * ls[l] + nabs * P_.xsec[l];
          }
          Real base[NM];
#pragma unroll
          for (int m = 0; m < NM; m++) {
            const Real tau = kap[m] * s;
            const Real p = m_exp<Real>(-tau);
            const Real c = ((double) tau < 1e-3) ? (Real(1.0) - Real(0.5) * tau) : MathB<Real>::divq_(Real(1.0) - p, tau);
            base[m] = ok ? c * P[m][j] * s : Real(0);
            P[m][j] *= p;
          }
#pragma unroll
          for (int l = 0; l < NL; l++) Tint[l] += base[TR::mult(l)] * (P_.weight[l] * ls[l]);
        }
#pragma unroll
        for (int l = 0; l < NL; l++) {
          Real t = Tint[l];
          t += __shfl_xor_sync(FULL, t, 1);
          t += __shfl_xor_sync(FULL, t, 2);
          t += __shfl_xor_sync(FULL, t, 4);
          if (t > s) t = s;                                             // :284-299
          if (act) {
            accB[l] += in[2 + NLOW + TR::upper(l)] * P_.A[l] * t / Real(1e9);   // :302-316
            acc_tsp[l] += (in[2 + TR::lower(l)] * P_.sigma[l] * (P_.norm[l] * nf)) * s;
            acc_tab[l] += (nabs * P_.xsec[l]) * s;
          }
        }
        if (act) {
#pragma unroll
          for (int l = 0; l < NLOW; l++) acc_col[l] += in[2 + l] * s;
        }
      }
    }
    j0 += LPR;

    if (have && j0 >= total) {
      if (sub == 0) {
#pragma unroll
        for (int l = 0; l < NL; l++) {
          out[(size_t) (0 * NL + l) * n_los_total + los] = accB[l];
          out[(size_t) (1 * NL + l) * n_los_total + los] = acc_tsp[l];
          out[(size_t) (2 * NL + l) * n_los_total + los] = (flagbits & 1) ? Real(-1.0) : acc_tab[l];   // exits_bottom
        }
#pragma unroll
        for (int l = 0; l < NLOW; l++) out[(size_t) (3 * NL + l) * n_los_total + los] = acc_col[l];
      }
      have = false;
    }
  }
}

template <class TR>
bool desc_matches(const b200rt_multiplet_desc &d) {
  if (d.n_lines != TR::NL || d.n_multiplets != TR::NM || d.n_lower != TR::NLOW || d.n_upper != TR::NUP ||
      d.n_lambda != TR::NLAM)
    return false;
  for (int l = 0; l < TR::NL; l++)
    if (d.multiplet_index[l] != TR::mult(l) || d.lower_level_index[l] != TR::lower(l) || d.upper_level_index[l] != TR::upper(l))
      return false;
  return true;
}

#define MULT_DISPATCH(kind, ...)                                           \
  switch (kind) {                                                          \
    case B200RT_MULT_O1026: { typedef TraitsO TR; __VA_ARGS__; } break;     \
    case B200RT_MULT_H_LYMAN: { typedef TraitsH TR; __VA_ARGS__; } break;   \
    case B200RT_MULT_H_SINGLET: { typedef TraitsS TR; __VA_ARGS__; } break; \
    default: return cudaErrorInvalidValue;                                 \
  }

} // namespace

int mult_check_desc(const b200rt_multiplet_desc &d) {
  switch (d.kind) {
    case B200RT_MULT_O1026: return desc_matches<TraitsO>(d) ? 0 : 1;
    case B200RT_MULT_H_LYMAN: return desc_matches<TraitsH>(d) ? 0 : 1;
    case B200RT_MULT_H_SINGLET: return desc_matches<TraitsS>(d) ? 0 : 1;
  }
  return 1;
}

template <class Real>
MultParams<Real> mult_params(const b200rt_multiplet_desc &d) {
  MultParams<Real> p;
  for (int l = 0; l < MULT_MAX_LINES; l++) {
    p.sigma[l] = (Real) d.line_sigma_total[l]; p.A[l] = (Real) d.line_A[l]; p.xsec[l] = (Real) d.absorber_xsec[l];
    p.offset[l] = (Real) d.offset[l]; p.norm[l] = (Real) d.norm[l]; p.weight[l] = (Real) d.weight[l];
    p.solar[l] = (Real) d.solar_flux[l]; p.pumped[l] = d.pumped[l];
  }
  for (int u = 0; u < MULT_MAX_UPPER; u++) p.decay[u] = (Real) d.upper_state_decay_rate[u];
  p.T_ref = (Real) d.T_ref; p.lambda_max = (Real) d.lambda_max;
  p.delta_lambda = 2 * p.lambda_max / (d.n_lambda - 1);     // O_1026_tracker.hpp:190
  return p;
}
template MultParams<double> mult_params<double>(const b200rt_multiplet_desc &);
template MultParams<float> mult_params<float>(const b200rt_multiplet_desc &);

template <class Real>
cudaError_t launch_mult_tables(const b200rt_multiplet_desc &d, MultView<Real> mv, int n_vox, cudaStream_t s) {
  const MultParams<Real> P = mult_params<Real>(d);
  MULT_DISPATCH(d.kind, {
    const int n = n_vox * LPR * Dim<TR>::NLP;
    mult_table_kernel<Real, TR><<<(n + 255) / 256, 256, 0, s>>>(mv, P, n_vox);
  });
  return cudaGetLastError();
}

template <class Real>
cudaError_t launch_mult_pack(const b200rt_multiplet_desc &d, MultView<Real> mv, int n_vox, cudaStream_t s) {
  MULT_DISPATCH(d.kind, { mult_pack_kernel<Real, TR><<<(n_vox + 255) / 256, 256, 0, s>>>(mv, n_vox); });
  return cudaGetLastError();
}

template <class Real>
cudaError_t launch_mult_influence(const b200rt_multiplet_desc &d, const GridView<Real> &g, MultView<Real> mv, int v_begin,
                                  int v_end, ListView<Real> lists, double *K, int *work_counter,
                                  unsigned long long *step_counter, cudaStream_t s) {
  const long long n = (long long) (v_end - v_begin) * g.n_rays;
  if (n <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), s);
  if (e != cudaSuccess) return e;
  const MultParams<Real> P = mult_params<Real>(d);
  const int threads = 128;
  const long long tasks = (n + RPW - 1) / RPW;
  long long blocks = (tasks + threads / 32 - 1) / (threads / 32);
  if (blocks > (long long) NUM_SMS * 4) blocks = (long long) NUM_SMS * 4;
  MULT_DISPATCH(d.kind, {
    mult_march_kernel<Real, TR, 0><<<(unsigned) blocks, threads, 0, s>>>(g, mv, P, v_begin, n, lists, nullptr, K, nullptr,
                                                                          nullptr, nullptr, work_counter, step_counter);
  });
  return cudaGetLastError();
}

template <class Real>
cudaError_t launch_mult_single_scattering(const b200rt_multiplet_desc &d, const GridView<Real> &g, MultView<Real> mv,
                                          ListView<Real> lists, const int *shadow, double *S0, double *tau_sp,
                                          double *tau_abs, int *work_counter, cudaStream_t s) {
  const long long n = g.n_vox;
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), s);
  if (e != cudaSuccess) return e;
  const MultParams<Real> P = mult_params<Real>(d);
  const int threads = 128;
  const long long tasks = (n + RPW - 1) / RPW;
  long long blocks = (tasks + threads / 32 - 1) / (threads / 32);
  if (blocks > (long long) NUM_SMS * 4) blocks = (long long) NUM_SMS * 4;
  MULT_DISPATCH(d.kind, {
    mult_march_kernel<Real, TR, 1><<<(unsigned) blocks, threads, 0, s>>>(g, mv, P, 0, n, lists, shadow, nullptr, S0, tau_sp,
                                                                          tau_abs, work_counter, nullptr);
  });
  return cudaGetLastError();
}

template <class Real>
cudaError_t launch_mult_brightness(const b200rt_multiplet_desc &d, const GridView<Real> &g, MultView<Real> mv,
                                   const Real *los_in, long long los_stride, long long first, long long count,
                                   ListView<Real> lists, int n_subsamples, Real *out, long long n_los_total, int *queue,
                                   const int *order, cudaStream_t s) {
  if (count <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(queue, 0, sizeof(int), s);
  if (e != cudaSuccess) return e;
  const MultParams<Real> P = mult_params<Real>(d);
  const int threads = 128;
  const size_t smem = GeomTables<Real>::doubles(g.n_rb, g.n_sb) * sizeof(Real);
  long long blocks = (count * LPR + threads - 1) / threads;
  if (blocks > (long long) NUM_SMS * 4) blocks = (long long) NUM_SMS * 4;
  MULT_DISPATCH(d.kind, {
    e = cudaFuncSetAttribute(mult_brightness_kernel<Real, TR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    mult_brightness_kernel<Real, TR><<<(unsigned) blocks, threads, smem, s>>>(g, mv, P, los_in, los_stride, first, count, lists,
                                                                               n_subsamples, out, n_los_total, queue, order);
  });
  return cudaGetLastError();
}

#define INST(Real)                                                                                                          \
  template cudaError_t launch_mult_tables<Real>(const b200rt_multiplet_desc &, MultView<Real>, int, cudaStream_t);          \
  template cudaError_t launch_mult_pack<Real>(const b200rt_multiplet_desc &, MultView<Real>, int, cudaStream_t);            \
  template cudaError_t launch_mult_influence<Real>(const b200rt_multiplet_desc &, const GridView<Real> &, MultView<Real>,   \
                                                   int, int, ListView<Real>, double *, int *, unsigned long long *,         \
                                                   cudaStream_t);                                                          \
  template cudaError_t launch_mult_single_scattering<Real>(const b200rt_multiplet_desc &, const GridView<Real> &,           \
                                                           MultView<Real>, ListView<Real>, const int *, double *, double *, \
                                                           double *, int *, cudaStream_t);                                  \
  template cudaError_t launch_mult_brightness<Real>(const b200rt_multiplet_desc &, const GridView<Real> &, MultView<Real>,  \
                                                    const Real *, long long, long long, long long, ListView<Real>, int,     \
                                                    Real *, long long, int *, const int *, cudaStream_t);
INST(double)
INST(float)

} // namespace b200rt
