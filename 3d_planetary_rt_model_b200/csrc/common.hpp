// common.hpp -- internal declarations shared by the translation units of
// lib3d_planetary_rt_b200.so.  Nothing here is part of the C ABI (include/b200rt.h).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>
#include "../../include/b200rt.h"

namespace b200rt {

constexpr int N_LAMBDA = 20;        // singlet_CFR_tracker::n_lambda (reference los_tracker.hpp:122)
constexpr int MAX_EMISSIONS = 2;    // observation_fit drives Ly alpha + Ly beta together
constexpr int NUM_SMS = 148;        // B200

// ------------------------------------------------------------------ device buffers
struct DevBuf {
  void *p = nullptr;
  size_t bytes = 0;
  cudaError_t ensure(size_t need) {
    if (need <= bytes && p) return cudaSuccess;
    if (p) { cudaFree(p); p = nullptr; bytes = 0; }
    if (need == 0) need = 16;
    cudaError_t e = cudaMalloc(&p, need);
    if (e == cudaSuccess) bytes = need;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
  template <class T> T *as() const { return static_cast<T *>(p); }
};

// page-locked host scratch for the small read-backs of a call (row margins, residuals, counters, flags).  A copy into
// PAGEABLE memory makes the runtime wait for the stream inside the call, holding a lock that stalls the launches of
// every other context of the process: measured on the 40x20 sweep, four contexts ran their solves strictly one after
// the other (1.2e3 solves/s with 1, 2 or 4 threads) until these read-backs went through page-locked memory.
struct PinnedBuf {
  void *p = nullptr;
  size_t bytes = 0;
  cudaError_t ensure(size_t need) {
    if (need <= bytes && p) return cudaSuccess;
    if (p) { cudaFreeHost(p); p = nullptr; bytes = 0; }
    if (need < 4096) need = 4096;
    cudaError_t e = cudaHostAlloc(&p, need, cudaHostAllocDefault);
    if (e == cudaSuccess) bytes = need;
    return e;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; bytes = 0; }
  template <class T> T *as() const { return static_cast<T *>(p); }
};

// ------------------------------------------------------------------ grid tables (device view)
// Everything the traversal, the interpolation and the ray construction read.
// All of it is computed on the host (grid_host.cpp) with the libm calls the
// reference makes, then uploaded once per b200rt_set_grid_sph.
template <class Real>
struct GridView {
  int n_rb, n_sb, n_vox, n_rays, cap;
  int pp;                  // 1 = plane_parallel_grid: boundaries are the planes z = rb[i], n_sb = 2 (no cones)
  const int *vox_map;      // voxel-origin rays: source voxel of local slot i is vox_map[i] (nullptr: v_begin + i);
                           // lets one launch cover the interleaved voxel shards of a multi-GPU build
  const Real *rb;          // [n_rb]   radial boundaries
  const Real *sph_R2;      // [n_rb]   (rb/1e9)^2            sphere::set_radius
  const Real *sb;          // [n_sb]   sza boundaries
  const Real *cone_cos;    // [n_sb-2] cos(sb[k+1])           cone::set_angle
  const Real *cone_cos2;   // [n_sb-2]
  const Real *pts_r;       // [n_rb-1]
  const Real *log_pts_r;   // [n_rb-1]
  const Real *pts_s;       // [n_sb-1]
  const Real *vox_z;       // [n_vox]  r*cos(t) of the voxel point   atmo_point::rtp
  const Real *vox_zn;      // [n_vox]  vox_z / pts_r: the IEEE quotient the cone intersections start from (cone::intersections)
  const double *col_ct;    // [n_sb-1] cos(pt.t) as the double libm call ptray makes
  const double *col_st;    // [n_sb-1] sin(pt.t)
  const Real *ray_cost;    // [n_rays] std::cos(ray.t)         atmo_ray::tp
  const Real *ray_sint;    // [n_rays]
  const double *ray_cp;    // [n_rays] cos(ray.p) (double call in ptray)
  const Real *ray_domega;  // [n_rays]
  const int *ray_mult;     // [n_rays] rays of the full set this one stands for (march view: 2 for a folded mirror pair,
                           // and ray_domega is already multiplied by it); nullptr: 1 (full view)
  // voxel-origin rays: the sphere crossings of a ray depend on (radial shell of its voxel, cos of its polar angle) only,
  // so their ordered, trimmed list is built once per (shell, polar-angle class) and shared by every voxel of the shell
  // and every azimuth (traverse.cu, sphere_table_kernel).  nullptr: every ray builds its own.
  int n_cls;               // distinct values of ray_cost
  const int *ray_cls;      // [n_rays] class of each ray
  const int *cls_ray;      // [n_cls]  one ray of each class
  const int *sph_hdr;      // [(n_rb-1) * n_cls][2]: kept entries (-1: this pair takes the general path), unused
  const Real *sph_de;      // [(n_rb-1) * n_cls]     distance of `end` (+inf: none)
  const Real *sph_d;       // [(n_rb-1) * n_cls][2 n_rb]
  const int *sph_i;        // [(n_rb-1) * n_cls][2 n_rb]
};

// boundary lists produced by the traversal kernel for a batch of rays: fixed stride
// `cap` per ray so that no prefix pass is needed; only the used part is ever touched.
template <class Real>
struct ListView {
  Real *dist;      // [n_rays_batch][cap]
  int *ent;        // [n_rays_batch][cap]   boundary::entering
  int *len;        // [n_rays_batch]        trimmed length (0 = ray misses the grid)
  int *flag;       // [n_rays_batch]        bit0 = exits_bottom, bit1 = capacity overflow
  int cap;
};

// explicit ray descriptors (sun-ward rays, lines of sight)
template <class Real>
struct RayList {
  const Real *r, *z, *t, *cost, *lz;
  const int *i_voxel;   // may be null => -1 (search for the origin voxel)
};

// per-emission tables (device view)
template <class Real>
struct EmissionView {
  const Real *T_ratio, *density, *dtau_species, *dtau_absorber;              // voxel averages
  const Real *T_ratio_pt, *density_pt, *dtau_species_pt, *dtau_absorber_pt;  // voxel points
  const Real *phi;        // [n_vox][N_LAMBDA] line shape exp(-lambda_i^2 T_ratio) of the averages
  const Real *mrec;       // [n_vox][4][5]{kappa, wratio}: march records (influence.cu)
  const Real *sourcefn;   // [n_vox]
  const Real *rec_pt;     // [n_vox][8] interleaved {T_ratio_pt, density_pt, dtau_species_pt, dtau_absorber_pt, S, pad}
  const Real *rec_avg;    // [n_vox][8] the same for the voxel averages (brightness_nointerp)
  Real branching, sigma_ref, g_factor;
};

// ------------------------------------------------------------------ host-side state
struct HostGrid {
  int n_rb = 0, n_sb = 0, n_vox = 0, n_rays = 0, cap = 0;
  bool pp = false;         // plane_parallel_grid (grid/grid_plane_parallel.hpp)
  std::vector<double> rb, sb, pts_r, pts_s, ray_t, ray_p, ray_domega;
};

struct Emission {
  bool defined = false, have_K = false, have_S = false;
  double branching = 1, T_ref = 0, sigma_ref = 0, g_factor = 0;
  double residual = -1;
  DevBuf tabs;     // 8 * n_vox Real
  DevBuf phi;      // n_vox * N_LAMBDA Real
  DevBuf mrec;     // n_vox * 2 * N_LAMBDA Real
  DevBuf K;        // n_vox^2 double, row major
  DevBuf S0, tau_sp, tau_abs;  // n_vox double
  DevBuf S;        // n_vox double (solution)
  DevBuf S_real;   // n_vox Real   (what the brightness kernel reads)
  DevBuf rec_pt, rec_avg;   // n_vox * 8 Real each: interleaved records for the brightness gathers
  bool rec_dirty = true;    // tables or S changed since the records were packed
};

// ------------------------------------------------------------------ multiplet CFR emission (multiplet.cu)
constexpr int MULT_MAX_LINES = B200RT_MAX_LINES, MULT_MAX_LOWER = 3, MULT_MAX_UPPER = 4;
constexpr int MULT_LPR = 8;      // lanes per ray / line of sight in the multiplet kernels
constexpr int MULT_REC = 12;     // Reals per voxel record of the multiplet brightness kernel: T, n_abs, n[3], S[4], pad

// numeric line parameters as the kernels take them (by value)
template <class Real>
struct MultParams {
  Real sigma[MULT_MAX_LINES], A[MULT_MAX_LINES], xsec[MULT_MAX_LINES], decay[MULT_MAX_UPPER];
  Real offset[MULT_MAX_LINES], norm[MULT_MAX_LINES], weight[MULT_MAX_LINES], solar[MULT_MAX_LINES];
  int pumped[MULT_MAX_LINES];
  Real T_ref, lambda_max, delta_lambda;
};

template <class Real>
struct MultView {
  const Real *T, *T_pt, *nabs, *nabs_pt;          // [n_vox]
  const Real *n[MULT_MAX_LOWER], *n_pt[MULT_MAX_LOWER];
  Real *rec_step;   // [n_vox][8][NLP][n_mult + n_lines]: kappa[m], weight*lineshape/kappa per line (voxel averages)
  Real *rec_org;    // [n_vox][8][NLP][n_lines]: sigma n0 / decay * lineshape(T0)   (origin factors of G)
  Real *rec_w0;     // [n_vox][8][NLP][n_lines]: weight * lineshape(T0)             (holstein_T_final)
  Real *tsv, *tav;  // [n_vox][n_lines]: line-centre optical depths per unit path
  const Real *S;    // [n_vox * n_upper] source function in Real
  Real *rec_pt, *rec_avg;   // [n_vox][MULT_REC] brightness records
};

struct Multiplet {
  bool defined = false, have_K = false, have_S = false, rec_dirty = true;
  b200rt_multiplet_desc d;
  double residual = -1;
  DevBuf tabs;                       // 10 * n_vox Real: T, T_pt, nabs, nabs_pt, n[3], n_pt[3]
  DevBuf rec_step, rec_org, rec_w0, tsv, tav;
  DevBuf K, S0, tau_sp, tau_abs, S;  // double: [n_el][n_el], [n_el], [n_vox*n_lines] x2, [n_el]
  DevBuf S_real, rec_pt, rec_avg;
};

enum Phase { PH_TRAVERSE = 0, PH_INFLUENCE = 1, PH_SOLVE = 2, PH_BRIGHTNESS = 3, PH_IPH = 4, PH_ORDER = 5,
             PH_LW_STRUCTURE = 6, PH_LW_VALUES = 7, PH_LW_APPLY = 8, PH_COUNT = 9 };

// line-of-sight weighting functions of the resident lines of sight (los_weights.cu, api_weights.cu): CSR shared by
// the emissions, values [n_em][nnz] in Real
struct LosWeights {
  bool valid = false;      // cleared by a re-grid, new emission tables or g-factors, new lines of sight
  long long nnz = 0;
  DevBuf row_ptr;          // [n_los + 1] long long
  DevBuf row_cnt;          // [n_los] int: row lengths of the count pass
  DevBuf col;              // [nnz] int
  DevBuf val;              // [n_em][nnz] Real
  DevBuf rec;              // [n_em][2][n_vox][8] Real: the brightness records of the tables with S = 0
  DevBuf scratch;          // scan tile sums, bitmaps of large grids
  DevBuf xy;               // operand and result of b200rt_los_weights_apply (double)
};

// Quemerais IPH model: tables and the constants of BACKGROUND (ipbackgroundCFR_fun.f:176-235), iph.cu
struct IphTable {
  bool loaded = false;
  int kmax = 0, lmax = 0;
  float ua = 0, dpi = 0, sig = 0, dtap = 0, sigmaf = 0, dinf_b = 0, dinf_o = 0;
  float a[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};   // wind-frame rotation A11..A33
  DevBuf dev;   // alt[kmax] (m) | ang[lmax] | DANS | SO(:,:,2) | SN(:,:,2)
  DevBuf io;    // u v w fln n_steps per line of sight
};

} // namespace b200rt

namespace b200rt { struct Group; }

struct b200rt_ctx {
  b200rt::Group *group = nullptr;   // set only on the handle b200rt_create_multi returns: it owns no device state, every
                                    // call fans out to the member contexts (one per device), device_group.cu
  int device = 0;
  int precision = B200RT_F64;
  cudaStream_t stream = nullptr;
  std::string err;

  bool have_grid = false;
  b200rt::HostGrid hg;
  b200rt::DevBuf grid_tables;       // one slab holding every GridView array
  void *grid_view = nullptr;        // heap GridView<Real> (host struct of device pointers): every ray
  void *march_view = nullptr;       // heap GridView<Real>: the same grid with mirror pairs of rays folded (influence builds)
  int n_rays_marched = 0;           // rays of the march view (a device group sizes its fan-out by them)
  b200rt::DevBuf sph_table;         // ordered sphere-crossing lists per (radial shell, polar-angle class), traverse.cu
  b200rt::DevBuf sun_rays;          // RayList arrays for the n_vox sun-ward rays + shadow flags
  std::vector<int> shadow;          // host copy of the shadow test per voxel

  int n_em = 0;
  b200rt::Emission em[b200rt::MAX_EMISSIONS];
  b200rt::Multiplet mult;           // set by b200rt_set_multiplet: the context then carries ONE multiplet emission

  // traversal scratch (one batch of rays)
  b200rt::DevBuf list_dist, list_ent, list_len, list_flag;
  long long batch_rays = 0;
  b200rt::DevBuf work_counter;      // 2 ints: dynamic work index, capacity-overflow flag
  b200rt::DevBuf step_counter;      // unsigned long long
  b200rt::PinnedBuf host_scratch;   // solve read-backs (margins, residuals)
  b200rt::PinnedBuf host_out;       // brightness results on their way to PAGEABLE caller arrays (b200rt_brightness)
  b200rt::PinnedBuf host_stage;     // small uploads / downloads of caller (pageable) arrays travel through here
  b200rt::DevBuf dev_stage;         // float builds: the doubles of an upload before they are narrowed on the device
  b200rt::PinnedBuf host_words;     // counters and flags: [0] overflow flag (int), [1] step / sub-step counter (u64)
  long long last_steps = 0;
  long long last_substeps = 0;      // line-of-sight sub-steps of the last singlet brightness call

  // lines of sight
  int n_los = 0;
  b200rt::DevBuf los_in;            // 9 * n_los Real: x y z r t lx ly lz cost
  b200rt::DevBuf los_out;           // n_em * 4 * n_los Real
  b200rt::DevBuf los_order;         // per batch: processing order of the lines of sight (longest first) + its bins
  bool los_done = false;

  // dense solve workspace
  b200rt::DevBuf lu, lu_dinv, lu_flag;
  cudaStream_t stream2 = nullptr;            // chain stream of the LU (diagonal-block inverse + panel), high priority
  cudaStream_t stream3 = nullptr;            // stream of the L-shaped update next to the diagonal, high priority
  std::vector<cudaEvent_t> lu_events;
  std::vector<cudaEvent_t> timer_events;     // PhaseTimer's pool: created on first use, reused by every call
  size_t timer_used = 0;
  // distributed solve (solve_krylov.cu): this context's exchange block (peers write into it), the work area, the source
  // voxel ranges the last influence call built (= the rows this rank multiplies), the round counter's last value
  b200rt::DevBuf kry_xchg, kry_work, kry_bp;   // kry_bp: the own rows of A M^-1 (right-preconditioned iteration)
  std::vector<std::pair<int, int>> built_ranges;
  unsigned long long kry_round_base = 0;
  int kry_last_iters = 0;
  bool solve_attrs_set = false;              // the LU kernels' dynamic shared memory limits were raised on this device
  cudaGraphExec_t lu_graph = nullptr;        // the factorisation + back substitution of one (np, workspace), replayed
  int lu_graph_np = 0, lu_graph_launches = 0;
  const void *lu_graph_A = nullptr, *lu_graph_dinv = nullptr;

  // row sink (multi-GPU): peer-memory address of the solving GPU's K; finished row batches are DMA'd there over
  // NVLink by the copy engines while the next batch is marched
  b200rt::DevBuf vox_map;                    // source voxels of an interleaved shard, ascending
  void *row_sink[2] = {nullptr, nullptr};
  int row_sink_n_vox[2] = {0, 0};            // the geometry a sink was named for: a re-grid clears it, a mismatch is an error
  cudaStream_t copy_stream = nullptr;
  cudaStream_t out_stream = nullptr;     // device -> host results of the pipelined host-buffer brightness
  cudaEvent_t ev_rows = nullptr;
  int row_push_batches = 4;                  // a rank's row range is marched in at least this many batches when a sink is set

  // timing
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  float phase_ms[b200rt::PH_COUNT] = {};
  int phase_launches[b200rt::PH_COUNT] = {};

  b200rt::IphTable iph;
  b200rt::LosWeights lw;
};

namespace b200rt {

inline int fail(b200rt_ctx *c, int code, const std::string &msg) {
  if (c) c->err = msg;
  return code;
}

#define B200RT_CUDA(ctx, call)                                                              \
  do {                                                                                      \
    cudaError_t e__ = (call);                                                               \
    if (e__ != cudaSuccess)                                                                 \
      return ::b200rt::fail(ctx, B200RT_ERR_CUDA,                                           \
                            std::string(#call) + ": " + cudaGetErrorString(e__));           \
  } while (0)

// ---- grid_host.cpp
template <class Real>
int upload_grid(b200rt_ctx *c);
template <class Real>
void make_grid_sph(int n_rb, int n_sb, int n_theta, int n_phi, const double *rb, int szamethod,
                   int raymethod, double *sb, double *pts_r, double *pts_s, double *ray_t,
                   double *ray_p, double *ray_domega);
template <class Real>
void make_grid_pp(int n_rb, int n_theta, const double *rb, double *pts_r, double *ray_t, double *ray_domega);
// mirror-pair fold of a ray set in Real (b200rt_fold_rays): rep[k] = the ray whose march stands for ray k; returns the
// number of rays marched
template <class Real>
int fold_rays(int n_rays, const double *ray_t, const double *ray_p, const double *ray_domega, int *rep);
template <class Real>
void los_from_MSO(int n, const double *loc, const double *dir, double *x, double *y, double *z,
                  double *r, double *t, double *lx, double *ly, double *lz, double *cost);

// ---- traverse.cu  (compiled with -fmad=false: decides voxel indices)
// fills the sphere-list table g points to (g.sph_* already carved, g.n_cls / ray_cls / cls_ray set); once per grid
template <class Real>
cudaError_t launch_sphere_table(const GridView<Real> &g, cudaStream_t s);
template <class Real>
cudaError_t launch_traverse_voxel_rays(const GridView<Real> &g, int v_begin, int v_end,
                                       ListView<Real> out, int *overflow_flag, cudaStream_t s);
template <class Real>
cudaError_t launch_traverse_list(const GridView<Real> &g, RayList<Real> rays, long long n,
                                 ListView<Real> out, int *overflow_flag, cudaStream_t s);

// ---- influence.cu
template <class Real>
cudaError_t launch_influence(const GridView<Real> &g, const EmissionView<Real> &em, int v_begin,
                             int v_end, ListView<Real> lists, double *K, int *work_counter,
                             unsigned long long *step_counter, cudaStream_t s);
template <class Real>
cudaError_t launch_single_scattering(const GridView<Real> &g, const EmissionView<Real> &em,
                                     ListView<Real> lists, const int *shadow, double *S0,
                                     double *tau_sp, double *tau_abs, int *work_counter, cudaStream_t s);
template <class Real>
cudaError_t launch_phi_table(const Real *T_ratio, const Real *dts, const Real *dta, int n_vox, Real *phi, Real *mrec,
                             cudaStream_t s);

// ---- brightness.cu
template <class Real>
cudaError_t launch_brightness(const GridView<Real> &g, const EmissionView<Real> *em, int n_em,
                              const Real *los_in, long long los_stride, long long first,
                              long long count, ListView<Real> lists, int n_subsamples, Real *out,
                              long long n_los_total, int *queue, unsigned long long *substep_counter,
                              const int *order, cudaStream_t s);
// longest-first processing order of the `count` lists (counting sort of their lengths): bins = 2 * (cap + 1) ints of
// scratch, order = count ints.  Returns cudaErrorInvalidValue when cap is too large for the shared-memory histogram.
// two emissions and few lines of sight: the brightness launch gives each (line of sight, emission) pair its own group
bool brightness_splits_emissions(int n_em, long long count);
long long brightness_resident_groups();   // 4-lane groups the machine holds at once
cudaError_t launch_los_order(const int *len, long long count, int cap, int *bins, int *order, cudaStream_t s);
constexpr int LOS_ORDER_MAX_CAP = 8000;
// em.sourcefn may be null: the records then carry S = 0
template <class Real>
cudaError_t launch_pack_records(const EmissionView<Real> &em, int n_vox, Real *rec_pt, Real *rec_avg, cudaStream_t s);

// ---- los_weights.cu  (compiled with -fmad=false: the structure and value passes must agree on every stencil)
// structure pass: col == nullptr counts the rows into row_cnt[first + t]; otherwise fills the columns at row_ptr[first + t].
// bitmap_scratch: lw_bitmap_scratch_bytes(n_vox, count) bytes (0: none needed)
size_t lw_bitmap_scratch_bytes(int n_vox, long long count);
template <class Real>
cudaError_t launch_lw_structure(const GridView<Real> &g, const Real *los_in, long long los_stride, long long first,
                                long long count, ListView<Real> lists, int n_subsamples, unsigned *bitmap_scratch,
                                int *row_cnt, const long long *row_ptr, int *col, cudaStream_t s);
// row_ptr[0..n] = exclusive scan of row_cnt[0..n); scratch: lw_scan_scratch_bytes(n) bytes
size_t lw_scan_scratch_bytes(long long n);
cudaError_t launch_lw_scan(const int *row_cnt, long long n, long long *row_ptr, long long *scratch, cudaStream_t s);
// value pass: val must be zero; *missing is set if a stencil voxel was not found in its row (an internal error)
template <class Real>
cudaError_t launch_lw_values(const GridView<Real> &g, const EmissionView<Real> *em, int n_em, const Real *los_in,
                             long long los_stride, long long first, long long count, ListView<Real> lists, int n_subsamples,
                             const long long *row_ptr, const int *col, Real *val, long long nnz, int *queue,
                             unsigned long long *substep_counter, const int *order, int *missing, cudaStream_t s);
// transpose 0: y[n_rows] = W x[n_vox]; 1: y[n_vox] = W^T x[n_rows]
template <class Real>
cudaError_t launch_lw_apply(const long long *row_ptr, const int *col, const Real *val, long long n_rows, int n_vox,
                            int transpose, const double *x, double *y, cudaStream_t s);

// ---- multiplet.cu
template <class Real>
MultParams<Real> mult_params(const b200rt_multiplet_desc &d);
int mult_check_desc(const b200rt_multiplet_desc &d);     // 0 if the index tables match the kind's compiled-in ones
template <class Real>
cudaError_t launch_mult_tables(const b200rt_multiplet_desc &d, MultView<Real> mv, int n_vox, cudaStream_t s);
template <class Real>
cudaError_t launch_mult_influence(const b200rt_multiplet_desc &d, const GridView<Real> &g, MultView<Real> mv, int v_begin,
                                  int v_end, ListView<Real> lists, double *K, int *work_counter,
                                  unsigned long long *step_counter, cudaStream_t s);
template <class Real>
cudaError_t launch_mult_single_scattering(const b200rt_multiplet_desc &d, const GridView<Real> &g, MultView<Real> mv,
                                          ListView<Real> lists, const int *shadow, double *S0, double *tau_sp,
                                          double *tau_abs, int *work_counter, cudaStream_t s);
template <class Real>
cudaError_t launch_mult_pack(const b200rt_multiplet_desc &d, MultView<Real> mv, int n_vox, cudaStream_t s);
template <class Real>
cudaError_t launch_mult_brightness(const b200rt_multiplet_desc &d, const GridView<Real> &g, MultView<Real> mv,
                                   const Real *los_in, long long los_stride, long long first, long long count,
                                   ListView<Real> lists, int n_subsamples, Real *out, long long n_los_total, int *queue,
                                   const int *order, cudaStream_t s);
// ---- grid_host.cpp: tracker constants of the reference (O_1026_tracker.hpp, H_multiplet_tracker*.hpp) in Real
template <class Real>
int multiplet_desc_init(int kind, b200rt_multiplet_desc *d);

// ---- iph.cu  (compiled with -fmad=false)
int iph_set_table(b200rt_ctx *c, int kmax, int lmax, int ninf, float temp, const float *alt_au, const float *ang,
                  const float *dans, const float *sot, const float *so, const float *sn, const float *dinf_cm3);
int iph_load_table(b200rt_ctx *c, const char *fname);
int iph_background(b200rt_ctx *c, float fs, float xpos, float ypos, float zpos, int n_los, const float *u1,
                   const float *v1, const float *w1, float *fln, int *n_steps);
int iph_model(b200rt_ctx *c, double g_lya, const double *marspos, int n_los, const double *ra, const double *dec,
              double *iph_kR);

// ---- b200rt_api.cu: the two calls a device group hands its members with a slice of the caller's arrays
int los_download_slice(b200rt_ctx *c, double *const dst[4], long long stride, long long offset);
int brightness_slice(b200rt_ctx *c, int n, const double *const src[9], int n_subsamples, double *const dst[4],
                     long long stride, long long offset);

// ---- device_group.cu: one handle, several devices of one process (b200rt_create_multi)
b200rt_ctx *group_primary(b200rt_ctx *g);
b200rt_ctx *group_owner(b200rt_ctx *g, int i_emission);   // the member that gathered (and solves) emission e's rows
b200rt_ctx *group_owner_K(b200rt_ctx *g, int e);   // ... with every row of K assembled there (gathers after a distributed build)
int group_forward(b200rt_ctx *g, int rc);      // rc of a call on the primary member; copies its error text on failure
int group_destroy(b200rt_ctx *g);
int group_synchronize(b200rt_ctx *g);
int group_set_grid_sph(b200rt_ctx *g, int n_rb, int n_sb, int n_rays, const double *rb, const double *sb, const double *pts_r,
                       const double *pts_s, const double *ray_t, const double *ray_p, const double *ray_domega);
int group_set_grid_pp(b200rt_ctx *g, int n_rb, int n_rays, const double *rb, const double *pts_r, const double *ray_t,
                      const double *ray_domega);
int group_set_singlet(b200rt_ctx *g, int e, int n_em, double branching, double T_ref, double sigma_ref, double gf,
                      const double *a0, const double *a1, const double *a2, const double *a3, const double *a4,
                      const double *a5, const double *a6, const double *a7);
int group_set_multiplet(b200rt_ctx *g, const b200rt_multiplet_desc *d, const double *a0, const double *a1, const double *a2,
                        const double *a3, const double *a4, const double *a5);
int group_set_g_factor(b200rt_ctx *g, int e, double gf);
int group_influence(b200rt_ctx *g, int n_ranges, const int *v_begin, const int *v_end);
int group_solve(b200rt_ctx *g);
int group_generate_S(b200rt_ctx *g);
int group_counts(b200rt_ctx *g, int which, long long *n);
int group_set_sourcefn(b200rt_ctx *g, int e, const double *S);
int group_los_upload(b200rt_ctx *g, int n, const double *x, const double *y, const double *z, const double *r, const double *t,
                     const double *lx, const double *ly, const double *lz, const double *cost);
int group_brightness_resident(b200rt_ctx *g, int n_subsamples);
int group_los_download(b200rt_ctx *g, double *B, double *tsp, double *tab, double *col);
int group_brightness(b200rt_ctx *g, int n, const double *const src[9], int n_subsamples, double *const dst[4]);
int group_los_weights(b200rt_ctx *g, int n_subsamples, long long *nnz);
int group_los_weights_download(b200rt_ctx *g, long long *row_ptr, int *col, double *val);
int group_los_weights_apply(b200rt_ctx *g, int e, int transpose, const double *x, double *y);
int group_traverse_los(b200rt_ctx *g, long long capacity, int *len, int *eb, int *entering, double *distance,
                       long long *n_entries);
int group_kernel_ms(b200rt_ctx *g, int phase, float *ms, int *n_launches);
int group_iph_load_table(b200rt_ctx *g, const char *fname);
int group_iph_set_table(b200rt_ctx *g, int kmax, int lmax, int ninf, float temp, const float *alt_au, const float *ang,
                        const float *dans, const float *sot, const float *so, const float *sn, const float *dinf_cm3);
int group_iph_background(b200rt_ctx *g, float fs, float xpos, float ypos, float zpos, int n_los, const float *u,
                         const float *v, const float *w, float *fln, int *n_steps);
int group_iph_model(b200rt_ctx *g, double g_lya, const double *marspos, int n_los, const double *ra, const double *dec,
                    double *iph_kR);

// ---- peaks.cu
int measure_fp64_peaks(b200rt_ctx *c, double *dfma_tflops, double *dmma_tflops);

// ---- solve_krylov.cu
namespace api {
int exchange_block(b200rt_ctx *c, void **dev_ptr);
int solve_distributed(b200rt_ctx *c, int rank, int world, void *const *blocks, bool reset_timer, int cta_cap = 0);
}
// ---- solve.cu
struct SolveResult { double residual; double min_margin; int launches; };
int solve_dense(b200rt_ctx *c, int n, const double *K, double branching, const double *S0,
                double *S, SolveResult *res);
template <class Real>
cudaError_t launch_convert(const double *src, Real *dst, long long n, cudaStream_t s);

} // namespace b200rt
