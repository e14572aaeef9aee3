/* b200rt.h -- C ABI of the B200-native hot path of planetarymike/3D_planetary_RT_model.
 *
 * The reference has no FFI layer: its seam is the set of member functions that
 * are declared in headers but defined only in src/RT_gpu.cu (pulled in under
 * __CUDACC__, RT_grid.hpp:328-331).  Each entry point below names the reference
 * interface it replaces (paths relative to the reference's src/).  A maintainer
 * binds them from the reference's own host classes as shown in INTEGRATION.md.
 *
 * Conventions
 *  - plain pointers and sizes only; every array is a caller-owned HOST buffer of
 *    doubles (a float `Real` build widens losslessly) unless the name ends in _dev;
 *  - the context owns all device memory persistently (the reference mallocs and
 *    frees inside every call, RT_gpu.cu:150-191,264-299);
 *  - every function returns a b200rt_status; b200rt_last_error() gives the text.
 *    Nothing ever calls exit() (the reference's checkCudaErrors does);
 *  - a context is not thread-safe: one per host thread / per GPU;
 *  - there is NO CPU fallback: without a CUDA device b200rt_create fails.
 */
#ifndef B200RT_H
#define B200RT_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200rt_ctx b200rt_ctx;

typedef enum {
  B200RT_OK = 0,
  B200RT_ERR_CUDA = 1,          /* a CUDA runtime call failed */
  B200RT_ERR_ARG = 2,           /* bad argument */
  B200RT_ERR_STATE = 3,         /* call order: grid / emission / source function not set */
  B200RT_ERR_CAPACITY = 4,      /* a ray produced more boundary crossings than 2*n_rb+n_sb
                                   (boundary_set::append only asserts, boundaries.hpp:153-158) */
  B200RT_ERR_NOT_DOMINANT = 5,  /* I - w K is neither strictly row diagonally dominant nor certifiably an M-matrix
                                   (K >= 0, rho(w K) < 1): elimination without row exchanges would be unsafe */
  B200RT_ERR_NOMEM = 6
} b200rt_status;

enum { B200RT_F64 = 0, B200RT_F32 = 1 };          /* arithmetic of the ray march: Real.hpp:9-27 */
enum { B200RT_ROW_MAJOR = 0, B200RT_COL_MAJOR = 1 }; /* EIGEN_ROWMAJOR or not, Real.hpp:41-53 */

/* ---- lifetime -------------------------------------------------------------------
 * replaces cudaSetDevice(0) + per-call cudaMalloc/cudaFree (RT_gpu.cu:143,257,190,299) */
int b200rt_create(int device, int precision, b200rt_ctx **ctx);
int b200rt_destroy(b200rt_ctx *ctx);
const char *b200rt_last_error(const b200rt_ctx *ctx);
int b200rt_device_count(void);
/* Several GPUs of ONE process behind one handle.  The reference's callers make one call per phase
 * (RT_grid::generate_S_gpu / brightness_gpu, RT_gpu.cu:255-309,138-192; above them
 * observation_fit::generate_source_function + brightness, observation_fit.cpp:122-169,491-516), so the handle fans
 * each call out itself and every other entry point of this header takes it unchanged:
 *   geometry, emission tables, source function: replicated on every device;
 *   b200rt_generate_S / b200rt_influence*:      source-voxel rows split into interleaved shards.  Grids of
 *                                               B200RT_KRYLOV_MIN_N (2048) voxels and more, every row in the call and
 *                                               at most B200RT_KRYLOV_MAX_N unknowns: the rows STAY on the devices that
 *                                               built them (singlet and multiplet emissions).  Smaller singlet grids: the
 *                                               devices write their finished row batches into the resident K of the
 *                                               device that solves that emission (emission e: device e mod n; one
 *                                               emission: the first device) over peer memory (copy engines, NVLink)
 *                                               while marching the next batch.  Smaller multiplet grids (no row sink
 *                                               for them): the first device builds every row;
 *   b200rt_solve:                               large grids: all devices together, each multiplying its own rows
 *                                               ("distributed solve" below), S resident everywhere afterwards; small
 *                                               grids: each emission's LU on its device, side by side, S handed over;
 *   b200rt_get_influence, b200rt_influence_dev: the assembled matrix on the first device (rows gathered on demand);
 *   b200rt_brightness*, b200rt_iph_*:           lines of sight split by index, results at their offsets in the
 *                                               caller's arrays; counters add up, b200rt_last_kernel_ms is the
 *                                               slowest device's time.
 * Work too small to pay for the fan-out stays on the first device (B200RT_GROUP_MIN_RAYS voxel rays marched -- a mirror
 * pair of rays folded by b200rt_fold_rays counts once --, default 262144;
 * B200RT_GROUP_MIN_LOS lines of sight, default 65536).  n_dev <= 0: every visible device; dev_ids NULL: 0..n_dev-1;
 * one device: a plain context, exactly b200rt_create; an id may repeat (several members on one device, as the sweep's
 * contexts per GPU).  b200rt_group_size: devices behind a handle (1 for a plain one). */
int b200rt_create_multi(int n_dev, const int *dev_ids, int precision, b200rt_ctx **ctx);
int b200rt_group_size(const b200rt_ctx *ctx);

/* ---- geometry -------------------------------------------------------------------
 * replaces RT_grid::RT_to_device() for grid_type = spherical_azimuthally_symmetric_grid
 * (RT_gpu.cu:8-40; members grid_spherical_azimuthally_symmetric.hpp:47-73, grid.hpp:32-45).
 * Arrays are the members the reference's setup_voxels()/setup_rays() filled:
 *   radial_boundaries[n_rb], sza_boundaries[n_sb], pts_radii[n_rb-1], pts_sza[n_sb-1],
 *   rays[i].t, rays[i].p, rays[i].domega  (i < n_rays).
 * Derived tables (sphere R, R^2: intersections.cpp:53-56; cone cos, cos^2: :103-109;
 * ray cos/sin: atmo_vec.cpp:172-181; voxel points: :41-49) are rebuilt on the host with
 * the same libm calls the reference makes, so traversal is bit-exact. */
int b200rt_set_grid_sph(b200rt_ctx *ctx, int n_rb, int n_sb, int n_rays,
                        const double *radial_boundaries, const double *sza_boundaries,
                        const double *pts_radii, const double *pts_sza,
                        const double *ray_theta, const double *ray_phi, const double *ray_domega);

/* host helper: what setup_voxels()/setup_rays() compute from the radial boundaries
 * (grid_spherical_azimuthally_symmetric.hpp:302-333,365-406).  szamethod 0 = uniform,
 * 1 = uniform_cos; raymethod 0 = gauss, 1 = uniform.  Outputs sized as above
 * (n_rays = n_theta*n_phi). */
int b200rt_make_grid_sph(int precision, int n_rb, int n_sb, int n_theta, int n_phi,
                         const double *radial_boundaries, int szamethod, int raymethod,
                         double *sza_boundaries, double *pts_radii, double *pts_sza,
                         double *ray_theta, double *ray_phi, double *ray_domega);

/* plane-parallel geometry: replaces RT_grid::RT_to_device() for grid_type = plane_parallel_grid
 * (grid/grid_plane_parallel.hpp:17-60; observation_fit uses <40, 7>, observation_fit.hpp:48-50,
 * generate_source_function.cpp <40, 6>, :85-93).  n_vox = n_rb-1; boundaries are the planes
 * z = radial_boundaries[i] (plane::intersections, intersections.cpp:25-46); voxel points sit on the
 * +z axis (:204); rays have phi = 0 (:219).  Source function only: the reference has no
 * interp_weights on this grid (:304-311), so b200rt_brightness* fails with B200RT_ERR_STATE.
 * make_grid_pp = what setup_voxels()/setup_rays() derive from the boundaries (:189-223). */
int b200rt_set_grid_pp(b200rt_ctx *ctx, int n_rb, int n_rays, const double *radial_boundaries,
                       const double *pts_radii, const double *ray_theta, const double *ray_domega);
int b200rt_make_grid_pp(int precision, int n_rb, int n_theta, const double *radial_boundaries,
                        double *pts_radii, double *ray_theta, double *ray_domega);

/* host helper, no device needed: the mirror-pair fold b200rt_set_grid_sph / _pp apply to the influence build.  On an
 * azimuthally symmetric grid the voxel-origin rays at phi and 2 pi - phi cross the same voxels over the same lengths, so
 * b200rt_influence* marches such a pair once and adds its contribution with twice the ray's domega.  Rays pair when
 * their uploaded cos/sin(theta), cos(phi) and domega are bit-equal, or (F64 only) when cos/sin(theta) and domega are
 * bit-equal, cos(phi) agrees to 1.8e-15 and sin(phi) has the opposite sign.  rep[n_rays]: the ray whose march stands for
 * ray k (k itself for a marched ray; a pair is represented by its lower index); n_marched: rays marched per voxel. */
int b200rt_fold_rays(int precision, int n_rays, const double *ray_theta, const double *ray_phi,
                     const double *ray_domega, int *rep, int *n_marched);

/* ---- emissions ------------------------------------------------------------------
 * replaces singlet_CFR::copy_to_device_influence / copy_to_device_brightness
 * (singlet_CFR.hpp:565-613) + emission_voxels::copy_to_device_* (emission_voxels.hpp:241-268).
 * Arrays are the protected per-voxel tables singlet_CFR::define() fills
 * (singlet_CFR.hpp:62-77,419-492), n_vox = (n_rb-1)*(n_sb-1) each; element order = voxel id. */
int b200rt_set_singlet(b200rt_ctx *ctx, int i_emission, int n_emissions,
                       double branching_ratio, double species_T_ref, double species_sigma_T_ref,
                       double emission_g_factor,
                       const double *species_T_ratio, const double *species_density,
                       const double *dtau_species, const double *dtau_absorber,
                       const double *species_T_ratio_pt, const double *species_density_pt,
                       const double *dtau_species_pt, const double *dtau_absorber_pt);
/* singlet_CFR::set_emission_g_factor, singlet_CFR.hpp:282-284 */
int b200rt_set_g_factor(b200rt_ctx *ctx, int i_emission, double g);

/* ---- multiplet emissions -----------------------------------------------------------
 * replaces multiplet_CFR_emission::copy_to_device_influence / copy_to_device_brightness
 * (emission/multiplet_CFR_emission.hpp:472-512) for the three multiplet emission types of the reference:
 *   B200RT_MULT_O1026     O_1026_emission      (emission/O_1026.hpp, O_1026_tracker.hpp)   6 lines, 3 multiplets
 *   B200RT_MULT_H_LYMAN   H_lyman_multiplet    (emission/H_lyman_multiplet.hpp, H_multiplet_tracker.hpp)  4 lines
 *   B200RT_MULT_H_SINGLET H_lyman_singlet      (emission/H_lyman_multiplet_test.hpp)       2 lines
 * The descriptor carries the tracker's static tables (CUDA_STATIC_ARRAY_MEMBERs and the constexpr Doppler-width
 * block, O_1026_tracker.hpp:17-216): b200rt_multiplet_desc_init fills it for `kind` in the arithmetic of
 * `precision`; offset = line_wavelength_offset / doppler_width_wavelength_reference, norm = line_shape_normalization
 * at T_ref, weight = tracker.weight().  solar_flux[line] / pumped[line]: compute_single_scattering assigns
 * singlescat(voxel, upper(line)) = flux n_lower sigma / decay * holstein_T_final[line] for pumped lines
 * (O_1026.hpp:111-129: the J=2 lines; H_lyman_multiplet.hpp:148-155: every line).
 * A context carries ONE multiplet emission (the reference's oxygen_RT / ly_multiplet_RT are RT_grid<., 1, .>,
 * observation_fit.hpp:93-125); b200rt_set_multiplet replaces any singlet emissions.  Per-voxel arrays are the
 * protected members multiplet_CFR_emission::define fills (:60-66): species_density[_pt] as [n_lower][n_vox].
 * In multiplet mode the shared entry points keep their meaning with these shapes (n_el = n_vox * n_upper, element
 * = voxel * n_upper + state, emission_voxels.hpp:32; voxel_vector.hpp:19-21):
 *   b200rt_get_solution: sourcefn, singlescat [n_el]; tau_*_single_scattering [n_vox * n_lines] (voxel major)
 *   b200rt_get_influence: [n_el][n_el];  b200rt_set_sourcefn: [n_el]
 *   b200rt_brightness / b200rt_los_download: brightness, tau_species_final, tau_absorber_final [n_lines][n_los];
 *                        species_col_dens [n_lower][n_los]   (O_1026_tracker.hpp:163-179) */
#define B200RT_MAX_LINES 6
enum { B200RT_MULT_O1026 = 0, B200RT_MULT_H_LYMAN = 1, B200RT_MULT_H_SINGLET = 2 };
typedef struct {
  int kind;
  int n_lines, n_multiplets, n_lower, n_upper, n_lambda;
  int multiplet_index[B200RT_MAX_LINES], lower_level_index[B200RT_MAX_LINES], upper_level_index[B200RT_MAX_LINES];
  double line_sigma_total[B200RT_MAX_LINES], line_A[B200RT_MAX_LINES], absorber_xsec[B200RT_MAX_LINES];
  double upper_state_decay_rate[B200RT_MAX_LINES];   /* indexed by upper state */
  double offset[B200RT_MAX_LINES], norm[B200RT_MAX_LINES], weight[B200RT_MAX_LINES];
  double T_ref, lambda_max;
  double solar_flux[B200RT_MAX_LINES];
  int pumped[B200RT_MAX_LINES];
} b200rt_multiplet_desc;
int b200rt_multiplet_desc_init(int kind, int precision, b200rt_multiplet_desc *desc);
int b200rt_set_multiplet(b200rt_ctx *ctx, const b200rt_multiplet_desc *desc,
                         const double *species_density, const double *species_density_pt,
                         const double *species_T, const double *species_T_pt,
                         const double *absorber_density, const double *absorber_density_pt);

/* ---- source function ------------------------------------------------------------
 * b200rt_generate_S replaces RT_grid::generate_S_gpu() (RT_gpu.cu:255-309): influence
 * kernel + single scattering + solve for every emission.  The two halves are exposed
 * separately so that rows can be sharded over GPUs (rows [v_begin, v_end) only). */
int b200rt_generate_S(b200rt_ctx *ctx);
int b200rt_influence(b200rt_ctx *ctx, int v_begin, int v_end);
/* the same for several ascending, disjoint source-voxel ranges in one call: the interleaved shards that balance the cost
 * of low-altitude (long rays through many voxels) and high-altitude rows across GPUs.  A multiplet context builds all
 * n_upper element rows of every voxel in the ranges. */
int b200rt_influence_ranges(b200rt_ctx *ctx, int n_ranges, const int *v_begin, const int *v_end);
/* RT_grid::solve_gpu, emission_voxels::solve_gpu: (I - w K) S = S0 per emission.  Two solvers behind it, both FP64 whatever
 * the context's Real: a block LU without row exchanges (FP64 tensor-core DMMA; the matrix is checked to be diagonally
 * dominant or an M-matrix first, B200RT_ERR_NOT_DOMINANT otherwise) and a right-preconditioned GMRES (see "distributed
 * solve" below; with one rank it is simply the faster solve of a large system: 4.0 ms against 5.8 ms at 5841 unknowns).
 * Grids of B200RT_KRYLOV_MIN_N (2048) voxels and more whose rows were all built by this context and whose system has at
 * most B200RT_KRYLOV_MAX_N unknowns (n_vox, or n_el = n_vox * n_upper for a multiplet) take the GMRES and fall back to the
 * LU if it does not converge; everything else takes the LU.  B200RT_SOLVER = lu | gmres overrides the size rule.
 * Either way b200rt_last_residual reports the true relative residual afterwards. */
int b200rt_solve(b200rt_ctx *ctx);
/* ray-voxel steps of the last b200rt_influence call as the reference counts them (one step = one
 * RT_grid::influence_update, RT_grid.hpp:90-105, covering all emissions).  A folded mirror pair (b200rt_fold_rays) is
 * marched once and counted for both of its rays. */
int b200rt_last_step_count(b200rt_ctx *ctx, long long *n_steps);
/* line-of-sight sub-steps integrated by the last singlet b200rt_brightness* call: sum over lines of sight of
 * (segments inside the grid) x (n_subsamples - 1), one sub-step = one update_tracker_brightness_interp of every
 * emission (RT_grid.hpp:273-293) */
int b200rt_last_substep_count(b200rt_ctx *ctx, long long *n_substeps);

/* replaces RT_grid::emissions_solved_to_host / emissions_influence_to_host
 * (RT_gpu.cu:62-84; emission_voxels.hpp:273-291).  Any pointer may be NULL.
 * K is the raw influence matrix (before the branching-ratio scaling of pre_solve). */
int b200rt_get_solution(b200rt_ctx *ctx, int i_emission, double *sourcefn, double *singlescat,
                        double *tau_species_single_scattering, double *tau_absorber_single_scattering);
int b200rt_get_influence(b200rt_ctx *ctx, int i_emission, int layout, double *influence_matrix);
/* sourcefn upload for brightness without a solve (copy_to_device_brightness, emission_voxels.hpp:257-268) */
int b200rt_set_sourcefn(b200rt_ctx *ctx, int i_emission, const double *sourcefn);
/* relative residual max|(I-wK)S-S0|/max|S0| of the last solve */
int b200rt_last_residual(b200rt_ctx *ctx, int i_emission, double *residual);

/* device-resident access for multi-GPU row exchange (pointer into ctx memory,
 * row-major [n_vox][n_vox] doubles / [n_vox] doubles); valid until destroy or re-grid */
int b200rt_influence_dev(b200rt_ctx *ctx, int i_emission, void **K_dev, void **S0_dev,
                         void **tau_species_ss_dev, void **tau_absorber_ss_dev);
int b200rt_sourcefn_dev(b200rt_ctx *ctx, int i_emission, void **S_dev);

/* ---- multi-GPU row exchange over peer memory ------------------------------------------
 * The reference has no multi-GPU path (single cudaSetDevice(0), RT_gpu.cu:143,257).  Influence rows shard by source
 * voxel (RT_grid.hpp:166-167: rows are independent); the one exchange of the pipeline puts every rank's rows into the
 * solving GPU's resident K.  One process per GPU: the solving rank exports a CUDA IPC handle of its K
 * (b200rt_ipc_export_influence, 64 bytes, passed to the other ranks by any host channel), the others open it
 * (b200rt_ipc_open -> a device pointer valid in their process) and name it as their row sink; from then on
 * b200rt_influence(v_begin, v_end) marches its range in >= 4 batches and DMAs each finished batch into the sink with
 * the copy engines over NVLink WHILE the next batch is marched (no SMs, no collective kernel), and returns when the
 * rows have landed.  A host barrier across ranks then releases the solve.  Singlet emissions only: a multiplet context
 * refuses b200rt_ipc_export_influence and b200rt_set_row_sink (its rows stay where they were built: distributed solve).
 * (This is the form for a solve by factorisation on one GPU; the distributed solve below needs no row exchange at all.) */
int b200rt_ipc_export_influence(b200rt_ctx *ctx, int i_emission, void *handle64);
int b200rt_ipc_open(b200rt_ctx *ctx, const void *handle64, void **peer_ptr);
int b200rt_ipc_close(b200rt_ctx *ctx, void *peer_ptr);
int b200rt_set_row_sink(b200rt_ctx *ctx, int i_emission, void *peer_K_dev);   /* NULL clears */

/* ---- distributed solve: the rows stay where they were built ---------------------------
 * The N-GPU form of RT_grid::solve_gpu.  Instead of gathering K on one GPU and factorising it there, every rank keeps
 * the rows its b200rt_influence / b200rt_influence_ranges call built (no row sink) and all ranks solve
 * (I - w K) S = S0 together by GMRES -- for a multiplet context (I - K) S = S0 over the n_el element rows, every rank
 * multiplying the n_upper rows of each voxel it built: one step is one product with K, each rank multiplies its own rows and writes its
 * piece of the result into every rank's EXCHANGE BLOCK over peer memory (NVLink), then every rank orthogonalises the
 * assembled vector redundantly -- bit-identical on all ranks -- so S ends up resident on every rank with no row gather,
 * no broadcast and no host barrier.  K is the kernel of a second-kind integral equation: the step count does not grow
 * with the grid (csrc/solve_krylov.cu).  Right preconditioner on spherical grids: the inverted diagonal blocks of I - wK
 * over runs of B200RT_KRYLOV_MAX_NR / n_upper radial voxels of one SZA column with all their states (one state and at
 * most 128 radial voxels: the whole column), whose entries every rank contributes for its rows in one more exchange round
 * and which every rank inverts redundantly; 38 steps instead of 71 on the 100x60 grid at 1e-13.
 *   b200rt_solve_exchange:    this context's exchange block (B200RT_KRYLOV_BLOCK_BYTES of device memory, allocated on
 *                             first use, alive until destroy): its device pointer (ranks of one process, peer access
 *                             enabled) and/or a CUDA IPC handle of it (64 bytes; other processes open it with
 *                             b200rt_ipc_open).  Either output may be NULL.
 *   b200rt_solve_distributed: blocks[q] = rank q's exchange block as addressable from THIS process, blocks[rank] = the
 *                             own one.  Every rank calls it, after its influence call on the same grid, the same number
 *                             of times (the blocks carry monotonic round counters).  On return every emission's S is
 *                             resident on every rank (b200rt_get_solution, b200rt_brightness*), b200rt_last_residual
 *                             is the true relative residual |S0 - (I - wK) S| / |S0| and b200rt_last_kernel_ms
 *                             (B200RT_PHASE_SOLVE) counts the launches.  The union of the ranks' rows must be every
 *                             voxel; a rank that never arrives is reported (B200RT_ERR_CUDA) after 20 s, no convergence
 *                             within 160 steps as B200RT_ERR_NOT_DOMINANT.  world = 1 is allowed (one GPU, GMRES
 *                             instead of the LU).  Singlet emissions: n_vox <= B200RT_KRYLOV_MAX_N; a multiplet:
 *                             n_el <= B200RT_KRYLOV_MAX_N (B200RT_ERR_CAPACITY beyond).
 * A device group (b200rt_create_multi) does this behind b200rt_solve / b200rt_generate_S for grids of
 * B200RT_KRYLOV_MIN_N (default 2048) voxels and more; smaller systems keep the LU on the owning device.
 * B200RT_KRYLOV_MAX_N = 24576 covers the H Lyman multiplet on the 100x60 grid (5841 voxels x 4 states = 23364).
 * Knobs: B200RT_KRYLOV_TOL (relative residual of the Krylov recurrence, default 1e-13), B200RT_KRYLOV_MAXIT,
 * B200RT_KRYLOV_PC=0 (no preconditioner). */
#define B200RT_KRYLOV_MAX_N 24576
#define B200RT_KRYLOV_MAX_WORLD 16
#define B200RT_KRYLOV_MAX_NR 128
#define B200RT_KRYLOV_BLOCK_BYTES (B200RT_KRYLOV_MAX_WORLD * 128 + 2 * B200RT_KRYLOV_MAX_N * 8 + (unsigned long long) B200RT_KRYLOV_MAX_N * B200RT_KRYLOV_MAX_NR * 8)
int b200rt_solve_exchange(b200rt_ctx *ctx, void **block_dev, void *ipc_handle64);
int b200rt_solve_distributed(b200rt_ctx *ctx, int rank, int world, void *const *blocks);
int b200rt_last_solve_steps(b200rt_ctx *ctx, int *n_steps);   /* GMRES steps of the last distributed solve */

/* ---- observations ---------------------------------------------------------------
 * host helper: observation::add_MSO_observation (observation.hpp:46-65) + atmo_point::xyz +
 * atmo_vector::ptxyz (atmo_vec.cpp:51-61,256-290): MSO position / look direction ->
 * the atmo_vector fields the march needs.  loc, dir: [n][3]; outputs [n] each. */
int b200rt_los_from_MSO(int precision, int n_los, const double *loc_MSO, const double *dir_MSO,
                        double *x, double *y, double *z, double *r, double *t,
                        double *line_x, double *line_y, double *line_z, double *cost);

/* replaces RT_grid::brightness_gpu(obs, n_subsamples) (RT_gpu.cu:138-192) and
 * observation::to_device/to_host (observation.hpp:211-254).  Inputs are the fields of
 * obs_vecs[i] (pt.{x,y,z,r,t}, line_{x,y,z}, ray.cost); outputs are the four tracker
 * members observation_fit reads (observation_fit.cpp:491-559), laid out [n_emissions][n_los].
 * n_subsamples = 0 -> brightness_nointerp (RT_grid.hpp:320-322); 1 is illegal (:237). */
int b200rt_brightness(b200rt_ctx *ctx, int n_los,
                      const double *x, const double *y, const double *z, const double *r, const double *t,
                      const double *line_x, const double *line_y, const double *line_z, const double *cost,
                      int n_subsamples,
                      double *brightness, double *tau_species_final, double *tau_absorber_final,
                      double *species_col_dens);
/* the same in three steps, for callers that keep lines of sight resident in HBM */
int b200rt_los_upload(b200rt_ctx *ctx, int n_los,
                      const double *x, const double *y, const double *z, const double *r, const double *t,
                      const double *line_x, const double *line_y, const double *line_z, const double *cost);
int b200rt_brightness_resident(b200rt_ctx *ctx, int n_subsamples);
int b200rt_los_download(b200rt_ctx *ctx, double *brightness, double *tau_species_final,
                        double *tau_absorber_final, double *species_col_dens);

/* ---- line-of-sight weighting functions -------------------------------------------------
 * The brightness of a singlet emission is linear in its source function: in RT_grid::brightness (RT_grid.hpp:233-299)
 * every sub-step adds S_interp * g * w / sigma_ref / sqrt(pi) / 1e9 * T_int, where S_interp = sum_k w_k S[idx_k] is the
 * 4-corner interpolation of S and T_int (clamped at tau_species_voxel) depends on the emission tables and the geometry
 * only.  So brightness_e = W_e S_e, with W_e a sparse n_los x n_vox matrix: contribution functions (where along each
 * line of sight the emission originates), the exact derivative d brightness / d S, and a cheap re-evaluation when only S
 * changes.  The IPH background is not part of W (it does not depend on S).
 *   b200rt_los_weights: builds W_e for every singlet emission on the lines of sight resident in the context
 *     (b200rt_los_upload), with b200rt_brightness's n_subsamples rule: 0 = one step per segment with the voxel-average
 *     tables (brightness_nointerp), 1 = illegal (B200RT_ERR_ARG), otherwise interpolated sub-steps.  It needs the grid
 *     and the emission tables, not a source function (it works before any solve).  *nnz (may be NULL) = stored entries.
 *     W[l, v] = sum over l's sub-steps, in march order, of w_k * gfac * T_int for every stencil corner k with idx_k == v
 *     (without interpolation: the current voxel with weight 1); gfac = g_factor * branching / sigma_ref / sqrt(pi) / 1e9,
 *     so W_e S_e is in kR.  Column v is stored in row l iff some sub-step of l reads v with a nonzero interpolation
 *     weight; columns of a row are ascending and unique; a stored value may be exactly 0 (e.g. zero density); a line of
 *     sight that misses the grid has an empty row.  The structure is shared by the emissions.  The values are a
 *     deterministic function of the inputs (two builds, and a device group against a plain context, give the same
 *     bytes).  In a float context they are accumulated in float and widened on download.
 *     b200rt_last_substep_count reports the sub-steps of the build; b200rt_last_kernel_ms: phase 6 = structure passes,
 *     7 = value pass (and 0 / 5 the traversal and ordering kernels it runs).
 *     Refused with B200RT_ERR_STATE: a multiplet context, a plane-parallel grid (no brightness there either), no lines
 *     of sight; with B200RT_ERR_NOMEM: device memory too small for the matrix.
 *   The matrix stays on the device until the next build; a re-grid, new emission tables or g-factors, or new lines of
 *   sight (b200rt_los_upload, b200rt_brightness) make it stale, and download / apply then return B200RT_ERR_STATE.
 *   b200rt_los_weights_download: CSR of the matrix: row_ptr[n_los + 1] (int64, row_ptr[0] = 0, row_ptr[n_los] = nnz),
 *     col[nnz] (voxel ids), val[n_emissions][nnz].  Any pointer may be NULL.
 *   b200rt_los_weights_apply: transpose 0: y[n_los] = W_e x[n_vox]; 1: y[n_vox] = W_e^T x[n_los], in double.  W x sums
 *     each row in a fixed order (the same bits every run; not those of a sequential sum).  W^T x adds with atomics: its
 *     last bits may vary between runs.  b200rt_last_kernel_ms phase 8 = the product kernel.
 * A device group splits the lines of sight by index, as for the brightness: every member builds the rows of its slice;
 * download stitches the rows in order, W x fills each member's slice of y, W^T x adds the members' n_vox partial
 * vectors on the host in member order. */
int b200rt_los_weights(b200rt_ctx *ctx, int n_subsamples, long long *nnz);
int b200rt_los_weights_download(b200rt_ctx *ctx, long long *row_ptr, int *col, double *val);
int b200rt_los_weights_apply(b200rt_ctx *ctx, int i_emission, int transpose, const double *x, double *y);

/* ---- interplanetary hydrogen background ---------------------------------------------
 * replaces quemerais_iph_model -> Fortran BACKGROUND (quemerais_IPH_model/iph_model_interface.cpp:19-82,
 * ipbackgroundCFR_fun.f:1-741).  The table file (fsm99td12v20t80 layout, :107-164) is parsed ONCE per
 * context (the Fortran re-reads it on every call); lines of sight are independent device threads
 * (the Fortran loop :295-320 is serial).  float32 like the Fortran.
 *   set_table: arrays as they stand in the file -- alt_au[kmax] (AU), ang[lmax] (deg), dans/sot[kmax][lmax],
 *              so/sn[ninf][kmax][lmax], dinf_cm3[ninf]; temp = TEMP of the header line.
 *   background: BACKGROUND's own arguments (fs = line-centre solar flux at 1 AU [ph cm-2 s-1 A-1], observer
 *              [AU, ecliptic], look vectors [ecliptic]); fln = xsn(2) in rayleigh; n_steps (may be NULL) =
 *              outer march steps per line of sight.
 *   model:     quemerais_iph_model's arguments (g factor at Mars, Mars ecliptic position [AU], RA/Dec [deg]);
 *              result in kR, Real = double.
 *   extinction: observation::update_iph_extinction (observation.hpp:144-154), host helper:
 *              out = (tau_absorber_final == -1) ? 0 : iph * exp(-tau_absorber_final). */
int b200rt_iph_load_table(b200rt_ctx *ctx, const char *filename);
int b200rt_iph_set_table(b200rt_ctx *ctx, int kmax, int lmax, int ninf, float temp, const float *alt_au,
                         const float *ang, const float *dans, const float *sot, const float *so, const float *sn,
                         const float *dinf_cm3);
int b200rt_iph_background(b200rt_ctx *ctx, float fs, float xpos, float ypos, float zpos, int n_los,
                          const float *u, const float *v, const float *w, float *fln, int *n_steps);
int b200rt_iph_model(b200rt_ctx *ctx, double g_lya, const double *mars_ecliptic_pos, int n_los,
                     const double *ra, const double *dec, double *iph_kR);
int b200rt_iph_extinction(int n, const double *iph_unextincted, const double *tau_absorber_final, double *iph_observed);

/* ---- traversal (parity surface) -------------------------------------------------
 * grid.ray_voxel_intersections (grid_spherical_azimuthally_symmetric.hpp:459-509) for the
 * voxel-origin rays of source voxels [v_begin, v_end) (ray order: voxel major, ray minor)
 * or for the resident lines of sight: trimmed boundary lists, concatenated.
 * len[i] entries per ray; entering = boundary::entering, distance = boundary::distance
 * (boundaries.hpp:15-21); exits_bottom as boundary_intersection_stepper (:334-349). */
int b200rt_traverse_voxel_rays(b200rt_ctx *ctx, int v_begin, int v_end, long long capacity,
                               int *len, int *exits_bottom, int *entering, double *distance,
                               long long *n_entries);
int b200rt_traverse_los(b200rt_ctx *ctx, long long capacity,
                        int *len, int *exits_bottom, int *entering, double *distance,
                        long long *n_entries);

/* ---- timing ---------------------------------------------------------------------
 * device time (CUDA events on the ctx stream) of the kernels of the last call:
 * phase 0 = traversal, 1 = influence march, 2 = solve, 3 = brightness march (the march launches alone),
 * 4 = IPH, 5 = the longest-first ordering kernels of the lines of sight (3 launches per batch),
 * 6 / 7 / 8 = line-of-sight weights: structure passes (count, scan, fill), value pass, products (b200rt_los_weights*) */
int b200rt_last_kernel_ms(b200rt_ctx *ctx, int phase, float *ms, int *n_launches);
int b200rt_synchronize(b200rt_ctx *ctx);
/* measured FP64 peaks of this device (TFLOP/s): plain DFMA and DMMA.8x8x4 (mma.sync m8n8k4.f64).
 * They are the roofline denominators of the march kernels and of the solve; the reference has
 * no counterpart (its timing is my_clock, src/my_clock.cpp:5-15). */
int b200rt_measure_fp64_peaks(b200rt_ctx *ctx, double *dfma_tflops, double *dmma_tflops);

#ifdef __cplusplus
}
#endif
#endif
