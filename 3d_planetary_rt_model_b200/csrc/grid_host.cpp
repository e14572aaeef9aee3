// grid_host.cpp -- host-side table construction (plain C++, no device code).
//
// The voxel traversal must be bit-exact against the reference CPU build, whose
// transcendental inputs come from the host libm.  So everything that feeds the
// traversal is computed HERE, with the same calls and the same operand types the
// reference uses, and shipped to the device; the device never recomputes a
// cos/sin/log/hypot that decides an index.
//
// Type rules reproduced (they matter for Real = float): a *std::*-qualified call
// on a Real uses the float overload, an unqualified call uses the double function
// and rounds on assignment (reference atmo_vec.cpp has no using-directives).
//
// Build with IEEE semantics: no -ffast-math, -ffp-contract=off.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <thread>
#include <vector>
#include "common.hpp"

namespace b200rt {

namespace {
template <class T>
size_t carve(size_t &off, size_t n) {
  off = (off + 15) & ~size_t(15);
  size_t at = off;
  off += n * sizeof(T);
  return at;
}

// the per-ray tables the traversal and the march read (atmo_ray::tp, atmo_vector::ptray), in Real
template <class Real>
struct RayTables {
  std::vector<Real> cost, sint, dom;
  std::vector<double> cp;
  std::vector<char> lower;   // sin(ray.p) < 0: the ray is the mirror image of one with sin(ray.p) > 0
  RayTables(int n, const double *ray_t, const double *ray_p, const double *ray_domega)
      : cost(n), sint(n), dom(n), cp(n), lower(n) {
    for (int k = 0; k < n; k++) {
      const Real t = (Real) ray_t[k], p = (Real) ray_p[k];
      cost[k] = std::cos(t);
      sint[k] = std::sin(t);
      cp[k] = ::cos((double) p);
      dom[k] = (Real) ray_domega[k];
      lower[k] = ::sin((double) p) < 0;
    }
  }
};

template <class T>
bool same_bits(const T &a, const T &b) { return std::memcmp(&a, &b, sizeof(T)) == 0; }

// cos(phi) of a mirror pair: phi and 2 pi - phi are each rounded once (ulp(2 pi) = 8.9e-16) before libm takes the
// cosine, so the two values differ by up to ~1e-15 (measured: 6 x 2^-53 at n_phi = 32, 8 x 2^-53 at n_phi = 12)
constexpr double MIRROR_COS_TOL = 0x1p-49;   // 1.8e-15
// Mirror pairs of voxel-origin rays.  Every voxel point lies in the phi = 0 half-plane of an azimuthally symmetric grid,
// so the rays at phi and 2 pi - phi of one voxel cross the same voxels over the same lengths: the traversal reads a ray
// only through cos(theta), sin(theta) and cos(phi) (traverse.cu ray_scalars), and the march adds domega * G.  A pair is
// marched once with multiplicity 2.  Rays pair when
//   - all four tables are bit-equal (both precisions: the two lists are then identical by construction), or
//   - in double only, cos(theta), sin(theta) and domega are bit-equal, cos(phi) agrees to MIRROR_COS_TOL and sin(phi)
//     has the opposite sign.  The lists of such a pair agree to ~1e-13 relative in distance, and K moves by at most
//     ~4e-8 relative per contribution on the 100x60 grid.  In float, line_z rounds differently often enough that the
//     lists of a near pair drift apart (segment lengths up to 100 % on that grid), so float folds bit-equal pairs only.
// The lower index represents the pair; every other ray, and every ray of a set without mirror symmetry, stays single.
template <class Real>
int fold_pairs(const RayTables<Real> &rt, int *rep) {
  const int n = (int) rt.cost.size();
  for (int k = 0; k < n; k++) rep[k] = k;
  int marched = 0;
  for (int k = 0; k < n; k++) {
    if (rep[k] != k) continue;
    marched++;
    for (int q = k + 1; q < n; q++) {
      if (rep[q] != q || !same_bits(rt.cost[k], rt.cost[q]) || !same_bits(rt.sint[k], rt.sint[q]) ||
          !same_bits(rt.dom[k], rt.dom[q]))
        continue;
      const bool exact = same_bits(rt.cp[k], rt.cp[q]);
      const bool mirror = sizeof(Real) == sizeof(double) && rt.lower[k] != rt.lower[q] &&
                          std::fabs(rt.cp[k] - rt.cp[q]) <= MIRROR_COS_TOL;
      if (exact || mirror) { rep[q] = k; break; }
    }
  }
  return marched;
}
} // namespace

template <class Real>
int fold_rays(int n_rays, const double *ray_t, const double *ray_p, const double *ray_domega, int *rep) {
  return fold_pairs<Real>(RayTables<Real>(n_rays, ray_t, ray_p, ray_domega), rep);
}
template int fold_rays<double>(int, const double *, const double *, const double *, int *);
template int fold_rays<float>(int, const double *, const double *, const double *, int *);

// Derived tables + upload.  Mirrors (reference src/):
//   sphere::set_radius      grid/intersections.cpp:53-56   R = rb/1e9, R2 = R*R
//   cone::set_angle         grid/intersections.cpp:103-109 cos(angle), cos^2
//   log_pts_radii           grid/grid_spherical_azimuthally_symmetric.hpp:302-305
//   atmo_point::rtp         atmo_vec.cpp:41-49             x = r sin t cos p, z = r cos t
//   atmo_ray::tp            atmo_vec.cpp:172-181           cost, sint
//   atmo_vector::ptray      atmo_vec.cpp:228-249           needs cos(pt.t), sin(pt.t), cos(ray.p)
//   RT_grid::get_single_scattering RT_grid.hpp:121-139 + atmo_vector::ptxyz atmo_vec.cpp:256-290
template <class Real>
int upload_grid(b200rt_ctx *c) {
  const HostGrid &h = c->hg;
  const int n_rb = h.n_rb, n_sb = h.n_sb, n_vox = h.n_vox, n_rays = h.n_rays;

  std::vector<Real> rb(n_rb), R2(n_rb), sb(n_sb), ccos(std::max(n_sb - 2, 1)), ccos2(std::max(n_sb - 2, 1)),
      pr(n_rb - 1), lpr(n_rb - 1), ps(n_sb - 1), vz(n_vox), vzn(n_vox);
  std::vector<double> ct(n_sb - 1), st(n_sb - 1);
  // sun-ward rays
  std::vector<Real> sr(n_vox), sz(n_vox), stt(n_vox), scost(n_vox), slz(n_vox);
  std::vector<int> sidx(n_vox);
  c->shadow.assign(n_vox, 0);

  const Real scale = 1e9;
  for (int i = 0; i < n_rb; i++) {
    rb[i] = (Real) h.rb[i];
    Real R = rb[i] / scale;
    R2[i] = R * R;
  }
  for (int i = 0; i < n_sb; i++) sb[i] = (Real) h.sb[i];
  for (int k = 0; k < n_sb - 2; k++) {
    Real ca = std::cos(sb[k + 1]);
    ccos[k] = ca;
    ccos2[k] = ca * ca;
  }
  for (int i = 0; i < n_rb - 1; i++) {
    pr[i] = (Real) h.pts_r[i];
    lpr[i] = std::log(pr[i]);
  }
  for (int j = 0; j < n_sb - 1; j++) {
    ps[j] = (Real) h.pts_s[j];
    ct[j] = ::cos((double) ps[j]);
    st[j] = ::sin((double) ps[j]);
  }
  const Real rmin = rb[0];
  for (int i = 0; i < n_rb - 1; i++)
    for (int j = 0; j < n_sb - 1; j++) {
      const int v = i * (n_sb - 1) + j;
      const Real r = pr[i], t = ps[j], p = 0.;
      const Real x = r * ::sin((double) t) * ::cos((double) p);
      const Real y = r * ::sin((double) t) * ::sin((double) p);
      const Real z = r * ::cos((double) t);
      vz[v] = z;
      vzn[v] = z / r;
      c->shadow[v] = (z < 0 && x * x + y * y < rmin * rmin) ? 1 : 0;
      // ptxyz(pt, 0, 0, 1): line = (0,0,1)/hypot(hypot(0,0),1)
      const Real mag = ::hypot(::hypot(0.0, 0.0), 1.0);
      const Real lx = Real(0.) / mag, ly = Real(0.) / mag, lz = Real(1.) / mag;
      const Real costx = lx * (x / r), costy = ly * (y / r), costz = lz * (z / r);
      sr[v] = r; sz[v] = z; stt[v] = t; sidx[v] = v;
      scost[v] = costx + costy + costz;
      slz[v] = lz;
    }
  const RayTables<Real> rt(n_rays, h.ray_t.data(), h.ray_p.data(), h.ray_domega.data());
  const std::vector<Real> &rcost = rt.cost, &rsint = rt.sint, &rdom = rt.dom;
  const std::vector<double> &rcp = rt.cp;

  // polar-angle classes of the rays: rays with bitwise equal cos(theta) cross every sphere at the same distances
  std::vector<int> rcls(n_rays), cls_ray;
  for (int k = 0; k < n_rays; k++) {
    int c_id = -1;
    for (size_t q = 0; q < cls_ray.size() && c_id < 0; q++)
      if (std::memcmp(&rcost[cls_ray[q]], &rcost[k], sizeof(Real)) == 0) c_id = (int) q;
    if (c_id < 0) { c_id = (int) cls_ray.size(); cls_ray.push_back(k); }
    rcls[k] = c_id;
  }
  const int n_cls = (int) cls_ray.size();
  // the table pays when classes are shared (n_phi rays per class); n_rb <= 128 is what the fast kernels cover
  const bool use_table = !h.pp && n_rb <= 128 && 2 * n_cls <= n_rays;
  const size_t n_pairs = (size_t) (n_rb - 1) * n_cls;

  // march view: the representative rays of the mirror-pair fold (fold_pairs) in ascending order, domega * multiplicity
  // (doubling is exact).  The first ray of a polar-angle class is always a representative, so every class keeps one.
  std::vector<int> rep(n_rays);
  const int n_fold = fold_pairs<Real>(rt, rep.data());
  std::vector<Real> fcost, fsint, fdom;
  std::vector<double> fcp;
  std::vector<int> fcls, fmult, fpos(n_rays, -1), fcls_ray(n_cls);
  for (int k = 0; k < n_rays; k++)
    if (rep[k] == k) {
      fpos[k] = (int) fcost.size();
      fcost.push_back(rcost[k]); fsint.push_back(rsint[k]); fcp.push_back(rcp[k]); fcls.push_back(rcls[k]);
      fdom.push_back(rdom[k]); fmult.push_back(1);
    } else {
      fdom[fpos[rep[k]]] += rdom[k];   // bit-equal to the representative's: exactly 2 domega
      fmult[fpos[rep[k]]] += 1;
    }
  for (int q = 0; q < n_cls; q++) fcls_ray[q] = fpos[cls_ray[q]];

  // one slab
  size_t off = 0;
  const size_t o_rb = carve<Real>(off, n_rb), o_R2 = carve<Real>(off, n_rb), o_sb = carve<Real>(off, n_sb),
               o_cc = carve<Real>(off, n_sb), o_cc2 = carve<Real>(off, n_sb), o_pr = carve<Real>(off, n_rb),
               o_lpr = carve<Real>(off, n_rb), o_ps = carve<Real>(off, n_sb), o_vz = carve<Real>(off, n_vox),
               o_ct = carve<double>(off, n_sb), o_st = carve<double>(off, n_sb),
               o_rc = carve<Real>(off, n_rays), o_rs = carve<Real>(off, n_rays),
               o_rcp = carve<double>(off, n_rays), o_rd = carve<Real>(off, n_rays),
               o_cls = carve<int>(off, n_rays), o_clr = carve<int>(off, n_cls), o_vzn = carve<Real>(off, n_vox),
               o_fc = carve<Real>(off, n_fold), o_fs = carve<Real>(off, n_fold), o_fcp = carve<double>(off, n_fold),
               o_fd = carve<Real>(off, n_fold), o_fcls = carve<int>(off, n_fold), o_fclr = carve<int>(off, n_cls),
               o_fm = carve<int>(off, n_fold);
  std::vector<char> slab(off + 16, 0);
  auto put = [&](size_t at, const void *src, size_t bytes) { std::memcpy(slab.data() + at, src, bytes); };
  put(o_rb, rb.data(), n_rb * sizeof(Real));       put(o_R2, R2.data(), n_rb * sizeof(Real));
  put(o_sb, sb.data(), n_sb * sizeof(Real));       put(o_cc, ccos.data(), (n_sb - 2) * sizeof(Real));
  put(o_cc2, ccos2.data(), (n_sb - 2) * sizeof(Real));
  put(o_pr, pr.data(), (n_rb - 1) * sizeof(Real)); put(o_lpr, lpr.data(), (n_rb - 1) * sizeof(Real));
  put(o_ps, ps.data(), (n_sb - 1) * sizeof(Real)); put(o_vz, vz.data(), n_vox * sizeof(Real));
  put(o_ct, ct.data(), (n_sb - 1) * sizeof(double)); put(o_st, st.data(), (n_sb - 1) * sizeof(double));
  put(o_rc, rcost.data(), n_rays * sizeof(Real));  put(o_rs, rsint.data(), n_rays * sizeof(Real));
  put(o_rcp, rcp.data(), n_rays * sizeof(double)); put(o_rd, rdom.data(), n_rays * sizeof(Real));
  put(o_vzn, vzn.data(), n_vox * sizeof(Real));
  put(o_cls, rcls.data(), n_rays * sizeof(int));   put(o_clr, cls_ray.data(), n_cls * sizeof(int));
  put(o_fc, fcost.data(), n_fold * sizeof(Real));  put(o_fs, fsint.data(), n_fold * sizeof(Real));
  put(o_fcp, fcp.data(), n_fold * sizeof(double)); put(o_fd, fdom.data(), n_fold * sizeof(Real));
  put(o_fcls, fcls.data(), n_fold * sizeof(int));  put(o_fclr, fcls_ray.data(), n_cls * sizeof(int));
  put(o_fm, fmult.data(), n_fold * sizeof(int));

  // the slab and, below, the sun-ward ray block each travel as one asynchronous copy out of page-locked staging (see
  // set_singlet_impl: copies out of pageable memory are staged by the runtime under a process-wide lock)
  const size_t rbytes = (size_t) n_vox * sizeof(Real);
  const size_t sun_bytes = 5 * rbytes + 2 * (size_t) n_vox * sizeof(int);
  B200RT_CUDA(c, c->host_stage.ensure(slab.size() + sun_bytes));
  B200RT_CUDA(c, c->grid_tables.ensure(slab.size()));
  std::memcpy(c->host_stage.p, slab.data(), slab.size());
  B200RT_CUDA(c, cudaMemcpyAsync(c->grid_tables.p, c->host_stage.p, slab.size(), cudaMemcpyHostToDevice, c->stream));

  if (c->grid_view) { ::operator delete(c->grid_view); c->grid_view = nullptr; }
  if (c->march_view) { ::operator delete(c->march_view); c->march_view = nullptr; }
  GridView<Real> *g = new GridView<Real>;
  char *base = static_cast<char *>(c->grid_tables.p);
  g->n_rb = n_rb; g->n_sb = n_sb; g->n_vox = n_vox; g->n_rays = n_rays; g->cap = h.cap; g->pp = h.pp ? 1 : 0;
  g->vox_map = nullptr;
  g->rb = (const Real *) (base + o_rb);          g->sph_R2 = (const Real *) (base + o_R2);
  g->sb = (const Real *) (base + o_sb);          g->cone_cos = (const Real *) (base + o_cc);
  g->cone_cos2 = (const Real *) (base + o_cc2);  g->pts_r = (const Real *) (base + o_pr);
  g->log_pts_r = (const Real *) (base + o_lpr);  g->pts_s = (const Real *) (base + o_ps);
  g->vox_z = (const Real *) (base + o_vz);       g->col_ct = (const double *) (base + o_ct);
  g->col_st = (const double *) (base + o_st);    g->ray_cost = (const Real *) (base + o_rc);
  g->ray_sint = (const Real *) (base + o_rs);    g->ray_cp = (const double *) (base + o_rcp);
  g->ray_domega = (const Real *) (base + o_rd);  g->ray_mult = nullptr;
  g->n_cls = n_cls;
  g->vox_zn = (const Real *) (base + o_vzn);
  g->ray_cls = (const int *) (base + o_cls);     g->cls_ray = (const int *) (base + o_clr);
  g->sph_hdr = nullptr; g->sph_de = nullptr; g->sph_d = nullptr; g->sph_i = nullptr;
  if (use_table) {
    size_t toff = 0;
    const size_t t_de = carve<Real>(toff, n_pairs), t_d = carve<Real>(toff, n_pairs * 2 * n_rb),
                 t_hdr = carve<int>(toff, n_pairs * 2), t_i = carve<int>(toff, n_pairs * 2 * n_rb);
    B200RT_CUDA(c, c->sph_table.ensure(toff + 16));
    char *tb = static_cast<char *>(c->sph_table.p);
    g->sph_de = (const Real *) (tb + t_de);  g->sph_d = (const Real *) (tb + t_d);
    g->sph_hdr = (const int *) (tb + t_hdr); g->sph_i = (const int *) (tb + t_i);
    B200RT_CUDA(c, launch_sphere_table<Real>(*g, c->stream));   // (same stream as the slab copy; the sync below covers it)
  }
  c->grid_view = g;
  GridView<Real> *f = new GridView<Real>(*g);   // shares everything but the rays (the sphere table included)
  f->n_rays = n_fold;
  f->ray_cost = (const Real *) (base + o_fc);    f->ray_sint = (const Real *) (base + o_fs);
  f->ray_cp = (const double *) (base + o_fcp);   f->ray_domega = (const Real *) (base + o_fd);
  f->ray_cls = (const int *) (base + o_fcls);    f->cls_ray = (const int *) (base + o_fclr);
  f->ray_mult = (const int *) (base + o_fm);
  c->march_view = f;
  c->n_rays_marched = n_fold;

  // sun-ward ray descriptors + shadow flags: [r | z | t | cost | lz](Real) [i_voxel | shadow](int)
  B200RT_CUDA(c, c->sun_rays.ensure(sun_bytes));
  char *hp = static_cast<char *>(c->host_stage.p) + slab.size();
  const void *srcs[5] = {sr.data(), sz.data(), stt.data(), scost.data(), slz.data()};
  for (int a = 0; a < 5; a++) std::memcpy(hp + a * rbytes, srcs[a], rbytes);
  std::memcpy(hp + 5 * rbytes, sidx.data(), n_vox * sizeof(int));
  std::memcpy(hp + 5 * rbytes + n_vox * sizeof(int), c->shadow.data(), n_vox * sizeof(int));
  B200RT_CUDA(c, cudaMemcpyAsync(c->sun_rays.p, hp, sun_bytes, cudaMemcpyHostToDevice, c->stream));
  B200RT_CUDA(c, cudaStreamSynchronize(c->stream));
  return B200RT_OK;
}
template int upload_grid<double>(b200rt_ctx *);
template int upload_grid<float>(b200rt_ctx *);

// Gauss-Legendre abscissas/weights, as the reference computes them
// (grid/gauss_legendre_quadrature.cpp:9-46, Numerical-Recipes gauleg)
template <class Real>
static void gauleg(const Real x1, const Real x2, std::vector<Real> &x, std::vector<Real> &w) {
  const Real strict_eps = sizeof(Real) == 4 ? Real(1e-5f) : Real(1e-10);
  Real z1, z, xm, xl, pp, p3, p2, p1;
  const int n = (int) x.size();
  const int m = (n + 1) / 2;
  xm = 0.5 * (x2 + x1);
  xl = 0.5 * (x2 - x1);
  for (int i = 0; i < m; i++) {
    z = std::cos(M_PI * (i + 0.75) / (n + 0.5));
    do {
      p1 = 1.0;
      p2 = 0.0;
      for (int j = 0; j < n; j++) {
        p3 = p2;
        p2 = p1;
        p1 = ((2 * j + 1) * z * p2 - j * p3) / (j + 1);
      }
      pp = n * (z * p1 - p2) / (z * z - 1.0);
      z1 = z;
      z = z1 - p1 / pp;
    } while (std::abs(z - z1) > strict_eps);
    x[i] = xm - xl * z;
    x[n - 1 - i] = xm + xl * z;
    w[i] = 2.0 * xl / ((1.0 - z * z) * pp * pp);
    w[n - 1 - i] = w[i];
  }
}

// What spherical_azimuthally_symmetric_grid::setup_voxels / setup_rays derive from the
// radial boundaries (grid_spherical_azimuthally_symmetric.hpp:302-333, 365-406;
// atmo_ray::set_ray_index atmo_vec.cpp:184-190).
template <class Real>
void make_grid_sph(int n_rb, int n_sb, int n_theta, int n_phi, const double *rb_in, int szamethod,
                   int raymethod, double *sb_out, double *pts_r, double *pts_s, double *ray_t,
                   double *ray_p, double *ray_domega) {
  const Real pi = M_PI;
  std::vector<Real> rb(n_rb), sb(n_sb);
  for (int i = 0; i < n_rb; i++) rb[i] = (Real) rb_in[i];
  for (int i = 0; i < n_rb - 1; i++) {
    Real p = ::sqrt(rb[i] * rb[i + 1]);
    pts_r[i] = p;
  }
  if (szamethod == 0) {
    Real sza_spacing = pi / (n_sb - 2.);
    for (int i = 0; i < n_sb; i++) sb[i] = (i - 0.5) * sza_spacing;
  } else {
    Real cs = 2.0 / (n_sb - 2.);
    sb[0] = -::acos(1.0 - 0.5 * cs);
    for (int i = 1; i < n_sb - 1; i++) sb[i] = ::acos(1.0 - (i - 0.5) * cs);
    sb[n_sb - 1] = pi + ::acos(1.0 - 0.5 * cs);
  }
  for (int i = 0; i < n_sb; i++) sb_out[i] = sb[i];
  for (int i = 0; i < n_sb - 1; i++) {
    Real p = 0.5 * (sb[i] + sb[i + 1]);
    pts_s[i] = p;
  }
  std::vector<Real> th(n_theta), wt(n_theta);
  if (raymethod == 0) {
    gauleg<Real>(0, pi, th, wt);
    for (int i = 0; i < n_theta; i++) wt[i] *= std::sin(th[i]);
  } else {
    Real theta_spacing = pi / (n_theta - 1);
    for (int i = 0; i < n_theta; i++) {
      th[i] = i * theta_spacing;
      if (i == 0 || i == n_theta - 1)
        wt[i] = 1 - std::cos(theta_spacing / 2);
      else
        wt[i] = (std::cos(th[i] - theta_spacing / 2) - std::cos(th[i] + theta_spacing / 2));
    }
  }
  Real phi_spacing = 2 * pi / n_phi;
  const Real quarter = 0.25;
  for (int i = 0; i < n_theta; i++)
    for (int j = 0; j < n_phi; j++) {
      const int k = i * n_phi + j;
      Real ph = (j + 0.5) * phi_spacing;
      Real dom = wt[i] * phi_spacing * quarter / pi;
      ray_t[k] = th[i];
      ray_p[k] = ph;
      ray_domega[k] = dom;
    }
}
template void make_grid_sph<double>(int, int, int, int, const double *, int, int, double *, double *, double *,
                                    double *, double *, double *);
template void make_grid_sph<float>(int, int, int, int, const double *, int, int, double *, double *, double *,
                                   double *, double *, double *);

// What plane_parallel_grid::setup_voxels / setup_rays derive from the radial boundaries
// (grid/grid_plane_parallel.hpp:189-223): geometric-mean voxel points, Gauss-Legendre theta on [0, pi]
// with weights w sin(theta), phi = 0, domega = w * 2pi / (4 pi) (atmo_ray::set_ray_index atmo_vec.cpp:184-190).
template <class Real>
void make_grid_pp(int n_rb, int n_theta, const double *rb_in, double *pts_r, double *ray_t, double *ray_domega) {
  const Real pi = M_PI;
  std::vector<Real> rb(n_rb);
  for (int i = 0; i < n_rb; i++) rb[i] = (Real) rb_in[i];
  for (int i = 0; i < n_rb - 1; i++) {
    Real p = ::sqrt(rb[i] * rb[i + 1]);
    pts_r[i] = p;
  }
  std::vector<Real> th(n_theta), wt(n_theta);
  gauleg<Real>(0, pi, th, wt);
  for (int i = 0; i < n_theta; i++) wt[i] *= std::sin(th[i]);
  const Real quarter = 0.25;
  for (int i = 0; i < n_theta; i++) {
    Real dom = wt[i] * (2 * pi) * quarter / pi;
    ray_t[i] = th[i];
    ray_domega[i] = dom;
  }
}
template void make_grid_pp<double>(int, int, const double *, double *, double *, double *);
template void make_grid_pp<float>(int, int, const double *, double *, double *, double *);

// ---------------------------------------------------------------- multiplet tracker constants
// The reference keeps these as constexpr members of its trackers, evaluated by the compiler in Real
// (O_1026_tracker.hpp:17-216; H_multiplet_tracker.hpp:17-173; H_multiplet_tracker_test.hpp:17-158; constants.hpp:14-22;
// constexpr_sqrt Real.hpp:63-82).  Restated in the same arithmetic so that a float build sees the float values.
namespace {
template <class Real>
Real newton_sqrt(Real x) {            // Detail::sqrtNewtonRaphson: iterate 0.5*(c + x/c) until it stops changing
  Real curr = x, prev = 0;
  while (curr != prev) {
    const Real next = 0.5 * (curr + x / curr);
    prev = curr;
    curr = next;
  }
  return curr;
}
template <class Real>
struct Doppler { Real wave, freq, norm; };
template <class Real>
Doppler<Real> doppler_block(Real ref_lambda_nm, Real ref_velocity) {
  const Real clight = 3e10;
  const Real one_over_sqrt_pi = ((Real) M_2_SQRTPI) / 2.0;
  Doppler<Real> d;
  d.wave = ref_lambda_nm * ref_velocity / clight;               // nm
  d.freq = 1.0 / (ref_lambda_nm * 1e-7) * ref_velocity;         // Hz (double expression, rounded to Real)
  d.norm = one_over_sqrt_pi / d.freq;                           // 1/Hz
  return d;
}
} // namespace

template <class Real>
int multiplet_desc_init(int kind, b200rt_multiplet_desc *d) {
  std::memset(d, 0, sizeof(*d));
  const Real kB = 1.38e-16, mH = 1.673e-24, line_f_coeff = 2.647e-2;
  const Real T_ref = 200, lambda_max = 4.0;
  d->kind = kind;
  d->T_ref = T_ref;
  d->lambda_max = lambda_max;
  if (kind == B200RT_MULT_O1026) {
    static const int mi[6] = {0, 1, 1, 2, 2, 2}, li[6] = {0, 1, 1, 2, 2, 2}, ui[6] = {0, 0, 1, 0, 1, 2}, lowJ[6] = {0, 1, 1, 2, 2, 2};
    static const double off[6] = {0.0, 4e-5, -4e-5, 8e-5, 1e-5, -9e-5};
    static const double A[6] = {4.22e7, 3.17e7, 5.71e7, 2.11e6, 1.91e7, 7.66e7};
    static const double f[6] = {2.01e-2, 5.02e-3, 1.51e-2, 2.00e-4, 3.01e-3, 1.69e-2};
    d->n_lines = 6; d->n_multiplets = 3; d->n_lower = 3; d->n_upper = 3; d->n_lambda = 21;
    const Real vel = newton_sqrt<Real>(2 * kB * T_ref / (16 * mH));
    const Doppler<Real> dw = doppler_block<Real>((Real) 102.57616, vel);
    const Real delta_lambda = 2 * lambda_max / (d->n_lambda - 1);
    for (int l = 0; l < 6; l++) {
      d->multiplet_index[l] = mi[l]; d->lower_level_index[l] = li[l]; d->upper_level_index[l] = ui[l];
      d->line_A[l] = (Real) A[l];
      d->line_sigma_total[l] = line_f_coeff * (Real) f[l];
      d->absorber_xsec[l] = (Real) 3.53e-17;
      d->offset[l] = (Real) ((Real) off[l] / dw.wave);
      d->norm[l] = dw.norm;
      d->weight[l] = (Real) (delta_lambda * dw.freq);
      d->pumped[l] = (lowJ[l] == 2);
    }
    d->upper_state_decay_rate[0] = (Real) (2.11e6 + 3.17e7 + 4.22e7 + 1.29e7 + 8.6e5 + 1.72e7);
    d->upper_state_decay_rate[1] = (Real) (1.91e7 + 5.71e7 + 2.32e7 + 7.74e6);
    d->upper_state_decay_rate[2] = (Real) (7.66e7 + 3.09e7);
    return B200RT_OK;
  }
  if (kind != B200RT_MULT_H_LYMAN && kind != B200RT_MULT_H_SINGLET) return B200RT_ERR_ARG;
  const bool single = (kind == B200RT_MULT_H_SINGLET);
  static const double off4[4] = {-2.70365e-4, 2.70365e-4, -5.703e-5, 5.703e-5};
  static const double A4[4] = {6.2648e8, 6.2649e8, 1.6725e8, 1.6725e8};
  static const double f4[4] = {0.2776, 0.13881, 5.2761e-2, 2.6381e-2};
  static const double x4[4] = {6.3e-20, 6.3e-20, 3.53e-17, 3.52e-17};
  d->n_lines = single ? 2 : 4; d->n_multiplets = 2; d->n_lower = 1; d->n_upper = single ? 2 : 4; d->n_lambda = 41;
  const Real vel = newton_sqrt<Real>(2 * kB * T_ref / mH);
  Doppler<Real> dw[2];
  if (single) {   // line_wavelength = {lyman_alpha_lambda*1e7, lyman_beta_lambda*1e7}: Real * double, rounded to Real
    const Real la = (Real) 121.6e-7, lb = (Real) 102.6e-7;
    dw[0] = doppler_block<Real>((Real) (la * 1e7), vel);
    dw[1] = doppler_block<Real>((Real) (lb * 1e7), vel);
  } else {
    dw[0] = doppler_block<Real>((Real) 121.5668237310, vel);
    dw[1] = doppler_block<Real>((Real) 102.572182505, vel);
  }
  const Real delta_lambda = 2 * lambda_max / (d->n_lambda - 1);
  for (int l = 0; l < d->n_lines; l++) {
    const int gi = single ? l : (l < 2 ? 0 : 1);   // Lyman alpha or beta
    d->multiplet_index[l] = gi; d->lower_level_index[l] = 0; d->upper_level_index[l] = l;
    if (single) {
      d->line_A[l] = (Real) (l == 0 ? 6.2648e8 : 1.6725e8);
      d->line_sigma_total[l] = line_f_coeff * (Real) (l == 0 ? 0.2776 + 0.13881 : 5.2761e-2 + 2.6381e-2);
      d->absorber_xsec[l] = (Real) (l == 0 ? 6.3e-20 : 3.52e-17);
      d->offset[l] = (Real) ((Real) 0.0 / dw[gi].wave);
      d->upper_state_decay_rate[l] = (Real) (l == 0 ? 6.2648e8 : 1.6725e8 + 2.2449e7);
    } else {
      d->line_A[l] = (Real) A4[l];
      d->line_sigma_total[l] = line_f_coeff * (Real) f4[l];
      d->absorber_xsec[l] = (Real) x4[l];
      d->offset[l] = (Real) ((Real) off4[l] / dw[gi].wave);
      d->upper_state_decay_rate[l] = (Real) (l == 0 ? 6.2648e8 : l == 1 ? 6.2649e8 : 1.6725e8 + 2.2449e7);
    }
    d->norm[l] = dw[gi].norm;
    d->weight[l] = (Real) (delta_lambda * dw[gi].freq);
    d->pumped[l] = 1;
  }
  return B200RT_OK;
}
template int multiplet_desc_init<double>(int, b200rt_multiplet_desc *);
template int multiplet_desc_init<float>(int, b200rt_multiplet_desc *);

// observation::add_MSO_observation (observation.hpp:46-65): model = (MSO_z, -MSO_y, MSO_x);
// atmo_point::xyz (atmo_vec.cpp:51-61); atmo_vector::ptxyz (atmo_vec.cpp:256-290).
template <class Real>
void los_from_MSO(int n, const double *loc, const double *dir, double *x, double *y, double *z, double *r,
                  double *t, double *lx, double *ly, double *lz, double *cost) {
  auto work = [=](int i0, int i1) {
    for (int i = i0; i < i1; i++) {
      const Real px = (Real) loc[3 * i + 2], py = -(Real) loc[3 * i + 1], pz = (Real) loc[3 * i + 0];
      const Real dx = (Real) dir[3 * i + 2], dy = -(Real) dir[3 * i + 1], dz = (Real) dir[3 * i + 0];
      const Real pr = ::hypot(::hypot((double) px, (double) py), (double) pz);
      const Real pt = ::acos((double) (pz / pr));
      const Real mag = ::hypot(::hypot((double) dx, (double) dy), (double) dz);
      const Real ux = dx / mag, uy = dy / mag, uz = dz / mag;
      const Real costx = ux * (px / pr), costy = uy * (py / pr), costz = uz * (pz / pr);
      x[i] = px; y[i] = py; z[i] = pz; r[i] = pr; t[i] = pt;
      lx[i] = ux; ly[i] = uy; lz[i] = uz;
      cost[i] = costx + costy + costz;
    }
  };
  unsigned nt = std::thread::hardware_concurrency();
  if (nt == 0) nt = 1;
  if (nt > 64) nt = 64;
  if (n < 20000) nt = 1;
  if (nt == 1) { work(0, n); return; }
  std::vector<std::thread> th;
  const int chunk = (n + (int) nt - 1) / (int) nt;
  for (unsigned k = 0; k < nt; k++) {
    const int i0 = (int) k * chunk, i1 = std::min(n, i0 + chunk);
    if (i0 < i1) th.emplace_back(work, i0, i1);
  }
  for (auto &q : th) q.join();
}
template void los_from_MSO<double>(int, const double *, const double *, double *, double *, double *, double *,
                                   double *, double *, double *, double *, double *);
template void los_from_MSO<float>(int, const double *, const double *, double *, double *, double *, double *,
                                  double *, double *, double *, double *, double *);

} // namespace b200rt
