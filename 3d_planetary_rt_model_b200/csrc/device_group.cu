// device_group.cu -- one handle, several GPUs of ONE process (b200rt_create_multi, include/b200rt.h).
//
// The reference drives a single device (cudaSetDevice(0), RT_gpu.cu:143,257).  Its callers -- RT_grid::generate_S_gpu /
// brightness_gpu and, above them, observation_fit::generate_source_function + brightness (observation_fit.cpp:122-169,
// 491-516) -- make ONE call per phase, so the way to give them N GPUs without touching their code is a context that
// fans each call out itself.  The handle b200rt_create_multi returns owns no device state: it holds one ordinary
// b200rt_ctx per device (member 0 = the solving GPU) and a host worker thread per further member, and every entry
// point of the C ABI dispatches here when it is handed such a handle (GROUP_DISPATCH in b200rt_api.cu):
//   geometry / emission tables / source function ... replicated on every member, in parallel;
//   influence rows ................................. split by source voxel into interleaved shards (the same cost
//                                                    balancing as the one-process-per-GPU path); every member names the
//                                                    primary's resident K as its row sink (plain peer access, no IPC:
//                                                    cudaDeviceEnablePeerAccess) and DMAs finished row batches there with
//                                                    its copy engines while it marches the next batch;
//   solve .......................................... on the primary; S is handed to the other members afterwards;
//   lines of sight (brightness, IPH) ............... split by index, no communication; results land in the caller's
//                                                    arrays at each member's offset.
// Work too small to pay for the fan-out stays on the primary (thresholds below, overridable by environment).
#include <algorithm>
#include <condition_variable>
#include <cstdlib>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>
#include "api_internal.hpp"

namespace b200rt {

namespace {

// one persistent host thread per member beyond the first: member calls synchronise their stream, so they have to be
// issued from different threads to overlap
class Worker {
 public:
  Worker() : th_([this] { loop(); }) {}
  ~Worker() {
    {
      std::lock_guard<std::mutex> lk(mu_);
      quit_ = true;
    }
    cv_.notify_all();
    th_.join();
  }
  void start(std::function<int()> job) {
    {
      std::lock_guard<std::mutex> lk(mu_);
      job_ = std::move(job);
      pending_ = true;
      done_ = false;
    }
    cv_.notify_all();
  }
  int wait() {
    std::unique_lock<std::mutex> lk(mu_);
    cv_.wait(lk, [this] { return done_; });
    return rc_;
  }

 private:
  void loop() {
    std::unique_lock<std::mutex> lk(mu_);
    for (;;) {
      cv_.wait(lk, [this] { return pending_ || quit_; });
      if (quit_) return;
      std::function<int()> job = std::move(job_);
      pending_ = false;
      lk.unlock();
      const int rc = job();
      lk.lock();
      rc_ = rc;
      done_ = true;
      cv_.notify_all();
    }
  }
  std::mutex mu_;
  std::condition_variable cv_;
  std::function<int()> job_;
  bool pending_ = false, done_ = true, quit_ = false;
  int rc_ = 0;
  std::thread th_;
};

long long env_ll(const char *name, long long dflt) {
  if (const char *e = getenv(name)) return atoll(e);
  return dflt;
}

}  // namespace

struct Group {
  std::vector<b200rt_ctx *> m;       // m[0] = primary (solving) device
  std::vector<Worker *> w;           // w[i] drives m[i], i >= 1 (w[0] unused)
  bool mult = false;
  int n_em = 0;
  // lines of sight: members [0, los_members) hold the slices [los_lo[i], los_lo[i + 1]) of the caller's arrays
  int los_members = 0;
  long long n_los = 0;
  std::vector<long long> los_lo;
  // bookkeeping of the last call(s), as b200rt_last_kernel_ms / *_count report them
  float phase_ms[PH_COUNT] = {0, 0, 0, 0, 0, 0};
  int phase_launches[PH_COUNT] = {0, 0, 0, 0, 0, 0};
  long long last_steps = 0, last_substeps = 0;
  // the member that gathered the rows of emission e in the last build and solves it (SURVEY 8(e): with several
  // emissions and several devices the dense solves run side by side, one emission per device)
  int owner[MAX_EMISSIONS] = {0, 0};
  // fan-out thresholds
  long long min_rays = 262144, min_los = 65536;
  int chunks_per_member = 8;
  // distributed solve (solve_krylov.cu): grids of kry_min_n voxels and more leave the rows on the members that built
  // them and all members solve together; `shard_b/e` remember who holds which rows (for the rare caller that asks for
  // the assembled matrix afterwards: rows_gathered)
  int kry_min_n = 2048;
  bool distributed = false, rows_gathered = true;
  std::vector<std::vector<int>> shard_b, shard_e;
};

namespace {

Group *G(b200rt_ctx *g) { return g->group; }

// run fn(i) for members [0, n_active): member 0 on the calling thread, the others on their workers; the first failure
// is reported on the group handle with the member's own message
int run_members(b200rt_ctx *g, int n_active, const std::function<int(int)> &fn) {
  Group *gr = G(g);
  for (int i = 1; i < n_active; i++) gr->w[i]->start([&fn, i] { return fn(i); });
  int rc = fn(0), bad = 0;
  for (int i = 1; i < n_active; i++) {
    const int r = gr->w[i]->wait();
    if (rc == B200RT_OK && r != B200RT_OK) { rc = r; bad = i; }
  }
  if (rc != B200RT_OK)
    g->err = "device " + std::to_string(gr->m[bad]->device) + ": " + gr->m[bad]->err;
  return rc;
}

int all(b200rt_ctx *g, const std::function<int(int)> &fn) { return run_members(g, (int) G(g)->m.size(), fn); }

void reset_phases(Group *gr) {
  for (int p = 0; p < PH_COUNT; p++) { gr->phase_ms[p] = 0; gr->phase_launches[p] = 0; }
}
// members ran side by side: a phase took as long as its slowest member; launches add up
void collect_phases(Group *gr, int n_active) {
  for (int p = 0; p < PH_COUNT; p++) {
    float ms = 0;
    int launches = 0;
    for (int i = 0; i < n_active; i++) {
      ms = std::max(ms, gr->m[i]->phase_ms[p]);
      launches += gr->m[i]->phase_launches[p];
    }
    gr->phase_ms[p] += ms;
    gr->phase_launches[p] += launches;
  }
}

void partition(long long n, int parts, int i, long long *lo, long long *hi) {
  const long long base = n / parts, rem = n % parts;
  *lo = i * base + std::min<long long>(i, rem);
  *hi = *lo + base + (i < rem ? 1 : 0);
}

int influence_rows(b200rt_ctx *g, int n_ranges, const int *vb, const int *ve) {
  Group *gr = G(g);
  b200rt_ctx *p = gr->m[0];
  if (!p->have_grid || (p->n_em < 1 && !p->mult.defined)) return fail(g, B200RT_ERR_STATE, "grid / emissions not set");
  long long n_rows = 0;
  int last_end = 0;
  for (int i = 0; i < n_ranges; i++) {
    if (vb[i] < last_end || ve[i] > p->hg.n_vox || vb[i] > ve[i])
      return fail(g, B200RT_ERR_ARG, "voxel ranges must be ascending, disjoint and inside the grid");
    last_end = ve[i];
    n_rows += ve[i] - vb[i];
  }
  const int n_mem = (int) gr->m.size();
  // large grids, every row of the grid in this build: the rows stay on their members and the solve is distributed
  const long long n_el = (long long) p->hg.n_vox * (p->mult.defined ? p->mult.d.n_upper : 1);
  const bool distributed = p->hg.n_vox >= gr->kry_min_n && n_el <= B200RT_KRYLOV_MAX_N && n_mem <= B200RT_KRYLOV_MAX_WORLD &&
                           n_rows == p->hg.n_vox;
  // the multiplet emissions have no row sink (b200rt.h: singlet emissions only): they fan out only for the distributed
  // solve; small builds do not pay for the fan-out.  Otherwise the build stays on the primary
  // (the work counted is the rays the build marches: mirror pairs folded, grid_host.cpp fold_pairs)
  const bool split = p->mult.defined ? distributed : (long long) n_rows * p->n_rays_marched >= gr->min_rays && n_rows >= 2 * n_mem;
  gr->distributed = false;
  gr->rows_gathered = true;
  if (!split) {
    for (int e = 0; e < MAX_EMISSIONS; e++) gr->owner[e] = 0;
    for (int e = 0; e < p->n_em && !p->mult.defined; e++) b200rt_set_row_sink(p, e, nullptr);
    const int rc = b200rt_influence_ranges(p, n_ranges, vb, ve);
    if (rc != B200RT_OK) { g->err = p->err; return rc; }
    collect_phases(gr, 1);
    gr->last_steps = p->last_steps;
    return B200RT_OK;
  }
  // interleaved shards: the flattened row list is cut into n_mem * chunks pieces dealt round-robin (rows from
  // low-altitude voxels cost more than rows from the outer corona; contiguous blocks would leave one member waiting)
  const int total = n_mem * gr->chunks_per_member;
  std::vector<std::vector<int>> rb(n_mem), re(n_mem);
  for (int c = 0; c < total; c++) {
    long long lo, hi;
    partition(n_rows, total, c, &lo, &hi);
    if (hi <= lo) continue;
    // flattened [lo, hi) -> voxel ranges
    long long base = 0;
    for (int i = 0; i < n_ranges && lo < hi; i++) {
      const long long len = ve[i] - vb[i];
      if (lo < base + len) {
        const long long a = std::max(lo, base), b = std::min(hi, base + len);
        if (b > a) {
          std::vector<int> &B = rb[c % n_mem], &E = re[c % n_mem];
          const int v0 = vb[i] + (int) (a - base), v1 = vb[i] + (int) (b - base);
          if (!E.empty() && E.back() == v0) E.back() = v1;     // adjacent pieces merge
          else { B.push_back(v0); E.push_back(v1); }
          lo = b;
        }
      }
      base += len;
    }
  }
  // emission e's rows are gathered on member e mod n_mem (one emission: the primary): every other member names that
  // member's resident K as its sink for e -- unless the solve is distributed
  gr->distributed = distributed;
  gr->rows_gathered = !gr->distributed;
  gr->shard_b = rb;
  gr->shard_e = re;
  for (int e = 0; e < MAX_EMISSIONS; e++) gr->owner[e] = (e < p->n_em && !gr->distributed) ? e % n_mem : 0;
  for (int i = 0; i < n_mem; i++)
    for (int e = 0; e < p->n_em; e++) {
      b200rt_ctx *own = gr->m[gr->owner[e]];
      const int rc = b200rt_set_row_sink(gr->m[i], e, (gr->distributed || gr->owner[e] == i) ? nullptr : own->em[e].K.p);
      if (rc != B200RT_OK) { g->err = gr->m[i]->err; return rc; }
    }
  const int rc = all(g, [&](int i) {
    return b200rt_influence_ranges(gr->m[i], (int) rb[i].size(), rb[i].data(), re[i].data());
  });
  if (rc != B200RT_OK) return rc;
  collect_phases(gr, n_mem);
  gr->last_steps = 0;
  for (int i = 0; i < n_mem; i++) gr->last_steps += gr->m[i]->last_steps;
  return B200RT_OK;
}

int solve_and_share(b200rt_ctx *g) {
  Group *gr = G(g);
  b200rt_ctx *p = gr->m[0];
  const int n_mem = (int) gr->m.size();
  const int n_e = p->mult.defined ? 1 : p->n_em;
  const size_t n_el = p->mult.defined ? (size_t) p->hg.n_vox * p->mult.d.n_upper : (size_t) p->hg.n_vox;
  if (gr->distributed) {
    // every member multiplies its own rows; S is resident on every member when the call returns
    std::vector<void *> blocks(n_mem, nullptr);
    for (int i = 0; i < n_mem; i++) {
      cudaSetDevice(gr->m[i]->device);
      if (int rc = api::exchange_block(gr->m[i], &blocks[i])) { g->err = gr->m[i]->err; return rc; }
    }
    // members that share a device (an id named several times) share its SMs: each one's resident grid shrinks so that all fit
    std::vector<int> cap(n_mem, 0);
    for (int i = 0; i < n_mem; i++) {
      int share = 0;
      for (int k = 0; k < n_mem; k++) share += gr->m[k]->device == gr->m[i]->device;
      cap[i] = share > 1 ? std::max(1, 2 * NUM_SMS / share) : 0;   // (0: the default, three CTAs per SM)
    }
    const int rc = run_members(g, n_mem, [&](int i) {
      cudaSetDevice(gr->m[i]->device);
      return api::solve_distributed(gr->m[i], i, n_mem, blocks.data(), true, cap[i]);
    });
    if (rc != B200RT_OK) return rc;
    collect_phases(gr, n_mem);
    return B200RT_OK;
  }
  bool spread = false;
  for (int e = 0; e < n_e; e++) spread = spread || gr->owner[e] != 0;
  if (!spread) {
    const int rc = b200rt_solve(p);
    if (rc != B200RT_OK) { g->err = p->err; return rc; }
    collect_phases(gr, 1);
  } else {
    // one emission per owner device, side by side
    const int rc = run_members(g, n_mem, [&](int i) {
      for (int e = 0; e < n_e; e++)
        if (gr->owner[e] == i)
          if (int r = api::solve_emission(gr->m[i], e)) return r;
      return (int) B200RT_OK;
    });
    if (rc != B200RT_OK) return rc;
    collect_phases(gr, n_mem);
  }
  // every member integrates lines of sight with the same source function
  std::vector<double> S(n_el);
  for (int e = 0; e < n_e; e++) {
    b200rt_ctx *own = gr->m[p->mult.defined ? 0 : gr->owner[e]];
    int rc = b200rt_get_solution(own, e, S.data(), nullptr, nullptr, nullptr);
    if (rc != B200RT_OK) { g->err = own->err; return rc; }
    rc = run_members(g, n_mem, [&](int i) { return gr->m[i] == own ? (int) B200RT_OK : b200rt_set_sourcefn(gr->m[i], e, S.data()); });
    if (rc != B200RT_OK) return rc;
  }
  return B200RT_OK;
}

}  // namespace

b200rt_ctx *group_primary(b200rt_ctx *g) { return G(g)->m[0]; }
// the member whose K holds every row of emission e.  After a distributed build the rows are still on the members that
// built them: they are copied to the primary here, once, for the caller that wants the assembled matrix
b200rt_ctx *group_owner_K(b200rt_ctx *g, int e) {
  Group *gr = G(g);
  if (gr->distributed && !gr->rows_gathered) {
    b200rt_ctx *p = gr->m[0];
    const bool mm = p->mult.defined;
    const size_t nu = mm ? p->mult.d.n_upper : 1, n = (size_t) p->hg.n_vox * nu;   // a voxel's rows: nu rows of n doubles
    const int n_K = mm ? 1 : p->n_em;
    auto K_of = [mm](b200rt_ctx *m, int em) { return mm ? m->mult.K.as<double>() : m->em[em].K.as<double>(); };
    for (size_t i = 1; i < gr->m.size(); i++)
      for (int em = 0; em < n_K; em++)
        for (size_t k = 0; k < gr->shard_b[i].size(); k++) {
          const size_t r0 = gr->shard_b[i][k] * nu, r1 = gr->shard_e[i][k] * nu;
          cudaMemcpyPeer(K_of(p, em) + r0 * n, p->device, K_of(gr->m[i], em) + r0 * n, gr->m[i]->device,
                         (r1 - r0) * n * sizeof(double));
        }
    cudaSetDevice(p->device);
    cudaDeviceSynchronize();
    gr->rows_gathered = true;
  }
  return group_owner(g, e);
}
b200rt_ctx *group_owner(b200rt_ctx *g, int e) {
  Group *gr = G(g);
  if (e < 0 || e >= MAX_EMISSIONS || gr->m[0]->mult.defined) return gr->m[0];
  return gr->m[gr->owner[e]];
}

int group_forward(b200rt_ctx *g, int rc) {
  if (rc != B200RT_OK) {      // the member that failed left its message; report the first non-empty one
    for (b200rt_ctx *m : G(g)->m) if (!m->err.empty()) { g->err = m->err; break; }
  }
  return rc;
}

int group_destroy(b200rt_ctx *g) {
  Group *gr = G(g);
  for (Worker *w : gr->w) delete w;           // joins
  for (size_t i = gr->m.size(); i-- > 1;) b200rt_destroy(gr->m[i]);   // the members that write into the primary's K go first
  if (!gr->m.empty()) b200rt_destroy(gr->m[0]);
  delete gr;
  g->group = nullptr;
  delete g;
  return B200RT_OK;
}

int group_synchronize(b200rt_ctx *g) {
  return all(g, [&](int i) { return b200rt_synchronize(G(g)->m[i]); });
}

int group_set_grid_sph(b200rt_ctx *g, int n_rb, int n_sb, int n_rays, const double *rb, const double *sb, const double *pts_r,
                       const double *pts_s, const double *ray_t, const double *ray_p, const double *ray_domega) {
  return all(g, [&](int i) {
    return b200rt_set_grid_sph(G(g)->m[i], n_rb, n_sb, n_rays, rb, sb, pts_r, pts_s, ray_t, ray_p, ray_domega);
  });
}

int group_set_grid_pp(b200rt_ctx *g, int n_rb, int n_rays, const double *rb, const double *pts_r, const double *ray_t,
                      const double *ray_domega) {
  return all(g, [&](int i) { return b200rt_set_grid_pp(G(g)->m[i], n_rb, n_rays, rb, pts_r, ray_t, ray_domega); });
}

int group_set_singlet(b200rt_ctx *g, int e, int n_em, double branching, double T_ref, double sigma_ref, double gf,
                      const double *a0, const double *a1, const double *a2, const double *a3, const double *a4,
                      const double *a5, const double *a6, const double *a7) {
  return all(g, [&](int i) {
    return b200rt_set_singlet(G(g)->m[i], e, n_em, branching, T_ref, sigma_ref, gf, a0, a1, a2, a3, a4, a5, a6, a7);
  });
}

int group_set_multiplet(b200rt_ctx *g, const b200rt_multiplet_desc *d, const double *a0, const double *a1, const double *a2,
                        const double *a3, const double *a4, const double *a5) {
  return all(g, [&](int i) { return b200rt_set_multiplet(G(g)->m[i], d, a0, a1, a2, a3, a4, a5); });
}

int group_set_g_factor(b200rt_ctx *g, int e, double gf) {
  for (b200rt_ctx *m : G(g)->m) b200rt_set_g_factor(m, e, gf);
  return B200RT_OK;
}

int group_influence(b200rt_ctx *g, int n_ranges, const int *v_begin, const int *v_end) {
  reset_phases(G(g));
  return influence_rows(g, n_ranges, v_begin, v_end);
}

int group_solve(b200rt_ctx *g) {
  reset_phases(G(g));
  return solve_and_share(g);
}

int group_generate_S(b200rt_ctx *g) {
  reset_phases(G(g));
  const int v0 = 0, v1 = G(g)->m[0]->hg.n_vox;
  if (int rc = influence_rows(g, 1, &v0, &v1)) return rc;
  return solve_and_share(g);
}

int group_counts(b200rt_ctx *g, int which, long long *n) {
  *n = which == 0 ? G(g)->last_steps : G(g)->last_substeps;
  return B200RT_OK;
}

int group_set_sourcefn(b200rt_ctx *g, int e, const double *S) {
  return all(g, [&](int i) { return b200rt_set_sourcefn(G(g)->m[i], e, S); });
}

// ---- lines of sight: split by index
namespace {
void slice_los(Group *gr, long long n) {
  const int n_mem = (int) gr->m.size();
  gr->los_members = (n >= gr->min_los && n >= n_mem) ? n_mem : 1;
  gr->n_los = n;
  gr->los_lo.assign(gr->los_members + 1, 0);
  for (int i = 0; i < gr->los_members; i++) {
    long long lo, hi;
    partition(n, gr->los_members, i, &lo, &hi);
    gr->los_lo[i] = lo;
    gr->los_lo[i + 1] = hi;
  }
}
}  // namespace

int group_los_upload(b200rt_ctx *g, int n, const double *x, const double *y, const double *z, const double *r, const double *t,
                     const double *lx, const double *ly, const double *lz, const double *cost) {
  Group *gr = G(g);
  if (n <= 0) return fail(g, B200RT_ERR_ARG, "there must be at least one observation to simulate");
  const double *src[9] = {x, y, z, r, t, lx, ly, lz, cost};
  for (auto p : src) if (!p) return fail(g, B200RT_ERR_ARG, "null line-of-sight array");
  slice_los(gr, n);
  return run_members(g, gr->los_members, [&](int i) {
    const long long lo = gr->los_lo[i];
    return b200rt_los_upload(gr->m[i], (int) (gr->los_lo[i + 1] - lo), x + lo, y + lo, z + lo, r + lo, t + lo, lx + lo,
                             ly + lo, lz + lo, cost + lo);
  });
}

int group_brightness_resident(b200rt_ctx *g, int n_subsamples) {
  Group *gr = G(g);
  if (gr->los_members <= 0) return fail(g, B200RT_ERR_STATE, "no lines of sight uploaded");
  reset_phases(gr);
  const int rc = run_members(g, gr->los_members, [&](int i) { return b200rt_brightness_resident(gr->m[i], n_subsamples); });
  if (rc != B200RT_OK) return rc;
  collect_phases(gr, gr->los_members);
  gr->last_substeps = 0;
  for (int i = 0; i < gr->los_members; i++) gr->last_substeps += gr->m[i]->last_substeps;
  return B200RT_OK;
}

int group_los_download(b200rt_ctx *g, double *B, double *tsp, double *tab, double *col) {
  Group *gr = G(g);
  if (gr->los_members <= 0) return fail(g, B200RT_ERR_STATE, "no brightness result to download");
  double *dst[4] = {B, tsp, tab, col};
  return run_members(g, gr->los_members, [&](int i) { return los_download_slice(gr->m[i], dst, gr->n_los, gr->los_lo[i]); });
}

int group_brightness(b200rt_ctx *g, int n, const double *const src[9], int n_subsamples, double *const dst[4]) {
  Group *gr = G(g);
  if (n <= 0) return fail(g, B200RT_ERR_ARG, "there must be at least one observation to simulate");
  for (int a = 0; a < 9; a++) if (!src[a]) return fail(g, B200RT_ERR_ARG, "null line-of-sight array");
  slice_los(gr, n);
  reset_phases(gr);
  const int rc = run_members(g, gr->los_members, [&](int i) {
    const long long lo = gr->los_lo[i];
    const double *s[9];
    for (int a = 0; a < 9; a++) s[a] = src[a] + lo;
    return brightness_slice(gr->m[i], (int) (gr->los_lo[i + 1] - lo), s, n_subsamples, dst, n, lo);
  });
  if (rc != B200RT_OK) return rc;
  collect_phases(gr, gr->los_members);
  gr->last_substeps = 0;
  for (int i = 0; i < gr->los_members; i++) gr->last_substeps += gr->m[i]->last_substeps;
  return B200RT_OK;
}

// parity surface: the members' lists one after the other = the lists of the whole set in order
int group_traverse_los(b200rt_ctx *g, long long capacity, int *len, int *eb, int *entering, double *distance,
                       long long *n_entries) {
  Group *gr = G(g);
  if (gr->los_members <= 0) return fail(g, B200RT_ERR_STATE, "no lines of sight uploaded");
  long long pos = 0;
  for (int i = 0; i < gr->los_members; i++) {
    long long got = 0;
    const long long lo = gr->los_lo[i];
    const int rc = b200rt_traverse_los(gr->m[i], capacity - pos, len + lo, eb + lo, entering + pos, distance + pos, &got);
    if (rc != B200RT_OK) { g->err = gr->m[i]->err; return rc; }
    pos += got;
  }
  if (n_entries) *n_entries = pos;
  return B200RT_OK;
}

int group_kernel_ms(b200rt_ctx *g, int phase, float *ms, int *n_launches) {
  if (ms) *ms = G(g)->phase_ms[phase];
  if (n_launches) *n_launches = G(g)->phase_launches[phase];
  return B200RT_OK;
}

// ---- interplanetary hydrogen: table on every member, lines of sight split by index
int group_iph_load_table(b200rt_ctx *g, const char *fname) {
  return all(g, [&](int i) { return b200rt_iph_load_table(G(g)->m[i], fname); });
}

int group_iph_set_table(b200rt_ctx *g, int kmax, int lmax, int ninf, float temp, const float *alt_au, const float *ang,
                        const float *dans, const float *sot, const float *so, const float *sn, const float *dinf_cm3) {
  return all(g, [&](int i) {
    return b200rt_iph_set_table(G(g)->m[i], kmax, lmax, ninf, temp, alt_au, ang, dans, sot, so, sn, dinf_cm3);
  });
}

int group_iph_background(b200rt_ctx *g, float fs, float xpos, float ypos, float zpos, int n_los, const float *u,
                         const float *v, const float *w, float *fln, int *n_steps) {
  Group *gr = G(g);
  const int n_mem = (int) gr->m.size();
  const int act = (n_los >= gr->min_los && n_los >= n_mem) ? n_mem : 1;
  reset_phases(gr);
  const int rc = run_members(g, act, [&](int i) {
    long long lo, hi;
    partition(n_los, act, i, &lo, &hi);
    return b200rt_iph_background(gr->m[i], fs, xpos, ypos, zpos, (int) (hi - lo), u + lo, v + lo, w + lo, fln + lo,
                                 n_steps ? n_steps + lo : nullptr);
  });
  if (rc == B200RT_OK) collect_phases(gr, act);
  return rc;
}

int group_iph_model(b200rt_ctx *g, double g_lya, const double *marspos, int n_los, const double *ra, const double *dec,
                    double *iph_kR) {
  Group *gr = G(g);
  const int n_mem = (int) gr->m.size();
  const int act = (n_los >= gr->min_los && n_los >= n_mem) ? n_mem : 1;
  reset_phases(gr);
  const int rc = run_members(g, act, [&](int i) {
    long long lo, hi;
    partition(n_los, act, i, &lo, &hi);
    return b200rt_iph_model(gr->m[i], g_lya, marspos, (int) (hi - lo), ra + lo, dec + lo, iph_kR + lo);
  });
  if (rc == B200RT_OK) collect_phases(gr, act);
  return rc;
}

}  // namespace b200rt

using namespace b200rt;

extern "C" {

int b200rt_create_multi(int n_dev, const int *dev_ids, int precision, b200rt_ctx **out) {
  if (!out || (precision != B200RT_F64 && precision != B200RT_F32)) return B200RT_ERR_ARG;
  *out = nullptr;
  const int visible = b200rt_device_count();
  if (visible <= 0) return B200RT_ERR_CUDA;                     // no CPU fallback
  std::vector<int> ids;
  if (n_dev <= 0) {                                              // every visible device
    for (int d = 0; d < visible; d++) ids.push_back(d);
  } else {
    for (int i = 0; i < n_dev; i++) {
      const int d = dev_ids ? dev_ids[i] : i;
      if (d < 0 || d >= visible) return B200RT_ERR_ARG;   // an id may repeat: several members on one device
      ids.push_back(d);
    }
  }
  if (ids.size() == 1) return b200rt_create(ids[0], precision, out);   // a plain context: nothing to fan out
  Group *gr = new (std::nothrow) Group;
  b200rt_ctx *g = new (std::nothrow) b200rt_ctx;
  if (!gr || !g) { delete gr; delete g; return B200RT_ERR_NOMEM; }
  gr->min_rays = env_ll("B200RT_GROUP_MIN_RAYS", gr->min_rays);
  gr->min_los = env_ll("B200RT_GROUP_MIN_LOS", gr->min_los);
  gr->chunks_per_member = (int) std::max(1LL, env_ll("B200RT_GROUP_CHUNKS", gr->chunks_per_member));
  gr->kry_min_n = (int) env_ll("B200RT_KRYLOV_MIN_N", gr->kry_min_n);
  g->group = gr;
  g->device = ids[0];
  g->precision = precision;
  for (int d : ids) {
    b200rt_ctx *m = nullptr;
    const int rc = b200rt_create(d, precision, &m);
    if (rc != B200RT_OK) { group_destroy(g); return rc; }
    gr->m.push_back(m);
    gr->w.push_back(gr->m.size() > 1 ? new Worker : nullptr);
  }
  // peer access in both directions between every pair: row batches are written into the primary's K by the members'
  // copy engines over NVLink.  Where a pair cannot map each other the copies still work (staged by the driver).
  for (int a : ids)
    for (int b : ids) {
      if (a == b) continue;
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, a, b) == cudaSuccess && can) {
        cudaSetDevice(a);
        const cudaError_t e = cudaDeviceEnablePeerAccess(b, 0);
        if (e != cudaSuccess) cudaGetLastError();   // cudaErrorPeerAccessAlreadyEnabled (another context of this process) is fine
      }
    }
  cudaSetDevice(ids[0]);
  *out = g;
  return B200RT_OK;
}

int b200rt_group_size(const b200rt_ctx *c) {
  if (!c) return 0;
  return c->group ? (int) c->group->m.size() : 1;
}

}  // extern "C"
