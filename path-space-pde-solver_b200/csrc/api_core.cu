// api_core.cu -- extern "C" entry points declared in include/pspde.h.
#include "api_common.h"
#include <mutex>
#include "rollout_tc_kernels.cuh"
#include "grad_kernels.cuh"
#include "grad_tc2_kernels.cuh"
#include "grad_tc_kernels.cuh"

thread_local char g_err[512] = "";
std::atomic<unsigned long long> g_launches{0};
unsigned long long* g_prof = nullptr;

// Index table of the shared weight image for the FP32-FMA kernels in 'outer' mode (RolloutParams::th_tbl): built on the host
// once per (device, network geometry) and cached (32 entries; a 33rd geometry evicts the oldest one -- cudaFree waits for the
// kernels that may still read it).  nullptr = allocation failure, reported by the launchers of the gradient kernels.
const int* pspde_theta_table(const NetGeom& g) {
  struct Entry { int dev, kind, L, time_mode, d, dims[PSPDE_MAXL + 1]; int* tbl; };
  static Entry cache[32];
  static int n_cache = 0;
  static std::mutex mu;
  int dev = 0;
#if !defined(PSPDE_EMULATE)
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
#endif
  std::lock_guard<std::mutex> lock(mu);
  for (int i = 0; i < n_cache; ++i) {
    const Entry& e = cache[i];
    bool same = e.dev == dev && e.kind == g.kind && e.L == g.L && e.time_mode == g.time_mode && e.d == g.d;
    for (int l = 0; same && l <= g.L; ++l) same = e.dims[l] == g.dims[l];
    if (same) return e.tbl;
  }
  static int n_evict = 0;
  int slot = n_cache;
  if (n_cache == 32) {
    slot = n_evict++ % 32;
#if defined(PSPDE_EMULATE)
    free(cache[slot].tbl);
#else
    cudaFree(cache[slot].tbl);
#endif
    cache[slot].tbl = nullptr; cache[slot].dev = -1;
  }
  const size_t n = 2 * (size_t)(g.w_floats >> 2);
  int* host = static_cast<int*>(malloc(n * sizeof(int)));
  if (!host) return nullptr;
  theta_table_fill(g, host);
  int* tbl = host;
#if !defined(PSPDE_EMULATE)
  tbl = nullptr;
  if (cudaMalloc(&tbl, n * sizeof(int)) != cudaSuccess || cudaMemcpy(tbl, host, n * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) {
    (void)cudaGetLastError();
    if (tbl) cudaFree(tbl);
    free(host);
    return nullptr;
  }
  free(host);
#endif
  Entry e;
  e.dev = dev; e.kind = g.kind; e.L = g.L; e.time_mode = g.time_mode; e.d = g.d; e.tbl = tbl;
  for (int l = 0; l <= PSPDE_MAXL; ++l) e.dims[l] = l <= g.L ? g.dims[l] : 0;
  cache[slot] = e;
  if (slot == n_cache) ++n_cache;
  return tbl;
}

// Must the zeta columns be written to the checkpoint?  Not when zeta = wY sqrt(dt) xi with in-kernel noise (adaptive process,
// no cotangent on Z_sum): the gradient kernel regenerates it from the Philox key (RolloutParams::ckpt_zeta).
// PSPDE_CKPT_ZETA=1 forces the columns into the checkpoint (A/B tests).
static int zeta_in_ckpt(const pspde_cfg* cfg, const float* wZ) {
  if (const char* e = getenv("PSPDE_CKPT_ZETA")) if (e[0] == '1') return 1;
  if (const char* e = getenv("PSPDE_GRAD_PATH")) if (!strcmp(e, "simt")) return 1;     // the FMA gradient kernel reads zeta
  return (cfg->noise_mode == PSPDE_NOISE_PHILOX && cfg->adaptive && !wZ) ? 0 : 1;
}
#if !defined(PSPDE_EMULATE)
// columns per (tile slot, step) of a checkpoint: [a0 (s0) | h1 | h2] and, only when it is written, zeta (s0)
static int ckpt_cols_of(const TcGeom& tg, int ckpt_zeta) { return ckpt_zeta ? tc_ckpt_cols(tg) : tg.s0 + 2 * tg.hp; }
#endif

// Forward rollout launch: the tensor-core kernel (rollout_tc_kernels.cuh) for the shape class it covers, else the
// FP32-FMA kernel.  PSPDE_FWD_PATH=simt forces the FMA kernel (A/B tests); PSPDE_FWD_PATH=tc makes an ineligible
// configuration an error.  *grid_out = number of CTAs launched (rows of stats_partial that were written); stats_room = bytes
// the caller's workspace holds for those rows.
static int launch_forward(const pspde_cfg* cfg, const Plan& pl, RolloutParams& p, bool tc_allowed, void* stream, int* grid_out,
                          size_t stats_room, int keep_tiles = 0) {
  const bool keep_ckpt = keep_tiles > 0;
#if !defined(PSPDE_EMULATE)
  TcGeom tg;
  const char* path = getenv("PSPDE_FWD_PATH");     // per call on purpose: the A/B tests switch paths inside one process
  const bool eligible = tc_allowed && cfg->N >= 1 && !(cfg->problem_flags & PSPDE_FLAG_DENSE_AB) && tc_geom(pl.g, cfg->d, tg);
  if (path && !strcmp(path, "tc") && !eligible) return fail(-6, "configuration is outside the tensor-core forward kernel's shape class");
  if (eligible && !(path && !strcmp(path, "simt"))) {
    const int n_tiles = (cfg->K_local + kTcP - 1) / kTcP;
    const int sms = pspde_sm_count();
    int grid = n_tiles < sms ? n_tiles : sms;
    apply_max_grid(grid);
    // every CTA writes 4 stats doubles at stats_partial[4 blockIdx.x]: checked against the caller's workspace (pl.stats_bytes
    // counts pl.grid CTAs of 64-path tiles, not this grid)
    if ((size_t)grid * 4 * sizeof(double) > stats_room)
      return fail(-7, "workspace too small for the forward's statistics (%zu < %zu)", stats_room, (size_t)grid * 4 * sizeof(double));
    p.n_tiles = n_tiles;
    if (keep_ckpt) { p.ckpt_zeta = zeta_in_ckpt(cfg, nullptr); p.ckpt_cols = ckpt_cols_of(tg, p.ckpt_zeta); p.ckpt_s0 = tg.s0;
                     p.tile0 = 0; p.ckpt_unit = 1; p.ckpt_tiles = keep_tiles; }
    const cudaError_t ce = keep_ckpt ? tc_launch_fwd_ckpt(p, tg, grid, (cudaStream_t)stream) : tc_launch(p, tg, grid, (cudaStream_t)stream);
    g_launches++;
    if (ce != cudaSuccess) return fail(-12, "tensor-core rollout launch failed: %s", cudaGetErrorString(ce));
    *grid_out = grid;
    return 0;
  }
#else
  (void)cfg; (void)tc_allowed;
#endif
  if (keep_ckpt) return fail(-6, "configuration is outside the checkpointing forward's shape class");
  *grid_out = pl.grid;
  return launch_rollout<512, false, 1>(pl, p, stream);
}

// ---- checkpointed detached backward: tensor-core forward (CKPT) + gradient accumulation, one wave of tiles at a time
struct CkptPlan {
  int n_tiles128, wave, cols, s0, grid_b;
  size_t ckpt_bytes, grad_bytes;
};

// Gradient accumulation from the checkpoint rows of n_ts (tile, step) pairs: the tensor-core kernel (grad_tc_kernels.cuh)
// for the shape class it covers, else the FP32-FMA kernel (grad_kernels.cuh).  PSPDE_GRAD_PATH=simt forces the FMA kernel
// (A/B tests), PSPDE_GRAD_PATH=tc makes an ineligible configuration an error.  `grid` = CTAs (<= n_ts; every CTA writes
// its own gradient partial).
static int launch_grad(const pspde_cfg* cfg, const Plan& pl, const RolloutParams& p, int grid, long long n_ts, void* stream, int* used_tc) {
  *used_tc = 0;
  if (n_ts < 1 || n_ts > 0x3fffffffLL) return fail(-6, "bad number of (tile, step) pairs for one gradient launch (%lld)", n_ts);
#if !defined(PSPDE_EMULATE)
  GradTcGeom gt;
  const char* path = getenv("PSPDE_GRAD_PATH");
  const bool eligible = grad_tc_geom(pl.g, cfg->d, p.ckpt_s0, gt);
  if (path && !strcmp(path, "tc") && !eligible) return fail(-6, "configuration is outside the tensor-core gradient kernel's shape class");
  if (eligible && !(path && !strcmp(path, "simt"))) {
    int flush_stages = kGtFlushStages;
    if (const char* e = getenv("PSPDE_GRAD_FLUSH_STAGES")) { const int v = atoi(e); if (v >= 1) flush_stages = v; }
    CUtensorMap tmap;
    // zeta regenerated in the kernel: one box of the activation rows per stage; else two boxes of cols / 2 rows
    if (!p.ckpt_zeta && gt.act_rows > 256) return fail(-6, "activation rows exceed one TMA box");
    if (grad_tc_tensor_map(gt, p.ckpt, n_ts, &tmap, p.ckpt_zeta ? 0 : gt.act_rows, p.ckpt_cols))
      return fail(-11, "cuTensorMapEncodeTiled failed for the checkpoint buffer");
    GradTc2Geom g2;
    // zeta from the Philox key: the kernel with the hidden cotangents on the tensor cores (PSPDE_GRAD_PATH=tc1: the older one)
    if (!p.ckpt_zeta && !(path && !strcmp(path, "tc1")) && grad_tc2_geom(pl.g, p.ckpt_s0, g2)) {
      if (cudaFuncSetAttribute(grad_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g2.total) != cudaSuccess)
        return fail(-11, "cudaFuncSetAttribute(%u B smem) failed", g2.total);
      grad_tc2_kernel<<<grid, kG2Threads, g2.total, (cudaStream_t)stream>>>(tmap, p, g2, (int)n_ts, flush_stages);
      g_launches++;
      if (const char* e = pspde_peek_error()) return fail(-12, "tensor-core gradient kernel (tc2) launch failed: %s", e);
      *used_tc = 2;
      return 0;
    }
    if (cudaFuncSetAttribute(grad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gt.total) != cudaSuccess)
      return fail(-11, "cudaFuncSetAttribute(%u B smem) failed", gt.total);
    grad_tc_kernel<<<grid, kGtThreads, gt.total, (cudaStream_t)stream>>>(tmap, p, gt, (int)n_ts, flush_stages);
    g_launches++;
    if (const char* e = pspde_peek_error()) return fail(-12, "tensor-core gradient kernel launch failed: %s", e);
    *used_tc = 1;
    return 0;
  }
#else
  (void)cfg;
#endif
  const int n_items = (int)(n_ts * (kCkP / kP));          // FMA kernel: work items of kP samples
  if (pl.T == 256) return pspde_launch_grad_256(pl, p, grid, n_items, stream);
  if (pl.T == 512) return pspde_launch_grad_512(pl, p, grid, n_items, stream);
  return fail(-13, "internal: no gradient kernel for T=%d", pl.T);
}

// floats of one CTA's gradient partial: weight-image layout (FMA kernel) or raw accumulator layout (tensor-core kernel)
static size_t grad_part_floats(const pspde_cfg* cfg, const Plan& pl, int s0) {
  size_t n = (size_t)pl.n_img_total;
#if !defined(PSPDE_EMULATE)
  GradTcGeom gt;
  if (grad_tc_geom(pl.g, cfg->d, s0, gt) && (size_t)(2 * 128 * gt.nB) > n) n = (size_t)(2 * 128 * gt.nB);
#else
  (void)cfg; (void)s0;
#endif
  return n;
}

// FP32-FMA kernels: weight-image partials of nparts CTAs -> grad_theta (reduce_grad_image_kernel)
static int reduce_grad_image(const Plan& pl, const RolloutParams& p, int nparts, float* grad_theta, void* stream) {
  if (!p.th_tbl) return fail(-13, "could not allocate the weight-image index table");
  const int w4 = pl.g.w_floats >> 2, tot = pl.n_sets * w4;
  PSPDE_LAUNCH(reduce_grad_image_kernel, (tot + 255) / 256, 256, 0, stream, p.grad_partial, nparts, pl.n_sets, w4, p.th_tbl,
               pl.g.n_params, grad_theta);
  g_launches++;
  if (const char* e = pspde_peek_error()) return fail(-12, "reduce_grad launch failed: %s", e);
  return 0;
}

static int reduce_grad(const pspde_cfg* cfg, const Plan& pl, const RolloutParams& p, int nparts, int used_tc, float* grad_theta, void* stream) {
  const int n = pl.n_theta_total;
#if !defined(PSPDE_EMULATE)
  if (used_tc) {
    GradTcGeom gt;
    grad_tc_geom(pl.g, cfg->d, p.ckpt_s0, gt);
    if (pspde_memset0(grad_theta, (size_t)n * sizeof(float), stream)) return fail(-12, "memset of grad_theta failed");
    const int per = 2 * 128 * gt.nB;
    if (used_tc == 2) {
      GradTc2Geom g2;
      grad_tc2_geom(pl.g, p.ckpt_s0, g2);
      reduce_grad_tc2_kernel<<<(per + 255) / 256, 256, 0, (cudaStream_t)stream>>>(pl.g, g2, p.grad_partial, nparts, grad_theta);
    } else {
      reduce_grad_tc_kernel<<<(per + 255) / 256, 256, 0, (cudaStream_t)stream>>>(pl.g, gt, p.grad_partial, nparts, grad_theta);
    }
    g_launches++;
    if (const char* e = pspde_peek_error()) return fail(-12, "reduce_grad_tc launch failed: %s", e);
    return 0;
  }
#else
  (void)cfg; (void)used_tc;
#endif
  (void)n;
  return reduce_grad_image(pl, p, nparts, grad_theta, stream);
}

#if !defined(PSPDE_EMULATE)
// true if the detached backward of cfg can take the checkpointed path (same shape class as the tensor-core forward)
static bool ckpt_plan(const pspde_cfg* cfg, const Plan& pl, TcGeom& tg, CkptPlan& cp) {
  if (cfg->N < 1 || (cfg->problem_flags & PSPDE_FLAG_DENSE_AB) || !tc_geom(pl.g, cfg->d, tg)) return false;
  const int sms = pspde_sm_count();
  cp.n_tiles128 = (cfg->K_local + kTcP - 1) / kTcP;
  // tiles per wave: two per SM (fewer launches, finer quantisation of the last wave) while the checkpoint buffer stays
  // below 12 GB, else one per SM up to 24 GB, else the configuration (very long horizons) takes the recompute kernel.
  // PSPDE_WAVE_TILES_PER_SM overrides the first choice.
  int per_sm = 2;
  if (const char* e = getenv("PSPDE_WAVE_TILES_PER_SM")) { const int v = atoi(e); if (v >= 1 && v <= 8) per_sm = v; }
  const size_t tile_bytes = (size_t)cfg->N * tc_ckpt_cols(tg) * kTcP * 4;
  auto wave_of = [&](int ps) { return cp.n_tiles128 < ps * sms ? cp.n_tiles128 : ps * sms; };
  if ((size_t)wave_of(per_sm) * tile_bytes > ((size_t)12 << 30)) per_sm = 1;
  if ((size_t)wave_of(per_sm) * tile_bytes > ((size_t)24 << 30)) return false;
  cp.wave = wave_of(per_sm);
  cp.cols = tc_ckpt_cols(tg);
  cp.s0 = tg.s0;
  const long long n_ts = (long long)cp.wave * cfg->N;
  cp.grid_b = n_ts < sms ? (int)n_ts : sms;
  // PSPDE_MAX_GRID caps the gradient CTAs but not the wave (still per_sm x SMs tiles): each CTA then runs more stages per
  // launch and flushes its accumulators many times, as at C5, at a K small enough for the fp64 oracle
  apply_max_grid(cp.grid_b);
  cp.ckpt_bytes = align256((size_t)cp.wave * cfg->N * cp.cols * kTcP * 4);
  cp.grad_bytes = align256((size_t)cp.grid_b * grad_part_floats(cfg, pl, tg.s0) * sizeof(float));
  return true;
}
#endif

// Single-rollout training step: the forward pass itself leaves the operand rows of ALL tiles (unit cotangents) and the
// gradient kernel applies dL/dY_N.  Needs the tensor-core shape class for both kernels and the adaptive (`-Z` drift)
// process with no cotangent on Z_sum (zeta = wY sqrt(dt) xi does not involve Z).  Returns the buffer size, 0 if ineligible.
static size_t fwd_ckpt_bytes(const pspde_cfg* cfg, const Plan& pl, size_t* tile_bytes = nullptr) {
#if !defined(PSPDE_EMULATE)
  TcGeom tg;
  GradTcGeom gt;
  for (const char* v : {"PSPDE_FWD_PATH", "PSPDE_BWD_PATH", "PSPDE_GRAD_PATH"})
    if (const char* e = getenv(v)) if (!strcmp(e, "simt")) return 0;
  if (cfg->N < 1 || !cfg->adaptive || (cfg->problem_flags & PSPDE_FLAG_DENSE_AB) || !tc_geom(pl.g, cfg->d, tg)) return 0;
  if (!grad_tc_geom(pl.g, cfg->d, tg.s0, gt)) return 0;
  const size_t n_tiles = (size_t)(cfg->K_local + kTcP - 1) / kTcP;
  const size_t tb = (size_t)cfg->N * ckpt_cols_of(tg, zeta_in_ckpt(cfg, nullptr)) * kTcP * 4;      // one 128-path tile; a multiple of 512 B
  if (tile_bytes) *tile_bytes = tb;
  return n_tiles * tb;
#else
  (void)cfg; (void)pl; (void)tile_bytes;
  return 0;
#endif
}

#if !defined(PSPDE_EMULATE)
// tiles [t_begin, n_tiles128) of the checkpointed detached backward: per wave, the tensor-core rollout that writes the operand
// rows (cotangents p.wY / p.wZ applied) into p.ckpt, then the gradient kernel; accumulates into p.grad_partial
static int run_waves(const pspde_cfg* cfg, const Plan& pl, RolloutParams& p, const TcGeom& tg, const CkptPlan& cp, int t_begin,
                     void* stream, int* used_tc) {
  // (the wave buffer is sized for rows WITH zeta columns; rows without them are simply shorter)
  p.ckpt_zeta = zeta_in_ckpt(cfg, p.wZ); p.ckpt_cols = ckpt_cols_of(tg, p.ckpt_zeta); p.ckpt_s0 = cp.s0; p.ckpt_unit = 0;
  const int sms = pspde_sm_count();
  for (int t0 = t_begin; t0 < cp.n_tiles128; t0 += cp.wave) {
    const int nt = cp.n_tiles128 - t0 < cp.wave ? cp.n_tiles128 - t0 : cp.wave;
    p.tile0 = t0; p.n_tiles = nt; p.ckpt_tiles = nt;
    int grid_f = nt < sms ? nt : sms;
    apply_max_grid(grid_f);
    const cudaError_t ce = tc_launch_t<true>(p, tg, grid_f, (cudaStream_t)stream);
    g_launches++;
    if (ce != cudaSuccess) return fail(-12, "tensor-core checkpoint rollout launch failed: %s", cudaGetErrorString(ce));
    const long long n_ts = (long long)nt * cfg->N;
    const int rc = launch_grad(cfg, pl, p, n_ts < cp.grid_b ? (int)n_ts : cp.grid_b, n_ts, stream, used_tc);
    if (rc) return rc;
  }
  return 0;
}
#endif

// u_L2 diagnostic descriptor (include/pspde.h) -> kernel parameters
static int set_udiag(const pspde_cfg* cfg, const pspde_udiag* diag, RolloutParams& p) {
  if (diag->mode < 0 || diag->mode > 2 || !diag->table || !diag->uL2) return fail(-8, "bad u_L2 diagnostic descriptor");
  if (diag->mode == 2 && (diag->nx1 < 1 || !(diag->dx > 0.f))) return fail(-8, "bad lookup-table geometry");
  if (diag->mode == 2 && (cfg->problem_flags & PSPDE_FLAG_DENSE_AB)) return fail(-8, "lookup diagnostic needs a diagonal problem");
  p.u_mode = diag->mode; p.u_tab = diag->table; p.u_nx1 = diag->nx1; p.u_d1 = diag->d1;
  p.u_xb = diag->xb; p.u_dx = diag->dx; p.uL2 = diag->uL2; p.u_quirk = diag->mode == 2 ? diag->quirk_path : -1;
  return 0;
}

extern "C" {

int pspde_abi_version(void) { return PSPDE_ABI_VERSION; }

int pspde_lv_cotangents(int K_local, double K_global, int moment, const float* Y_N, const float* gX, const double* stats,
                        float* wY, double* out3, void* stream) {
  if (K_local < 1 || !(K_global >= 1.0) || !Y_N || !gX || !stats || !wY || !out3) return fail(-1, "bad arguments");
  PSPDE_LAUNCH(lv_cotangents_kernel, (K_local + 255) / 256, 256, 0, stream, K_local, K_global, moment, Y_N, gX, stats, wY, out3);
  g_launches++;
  if (const char* e = pspde_peek_error()) return fail(-12, "lv_cotangents launch failed: %s", e);
  return 0;
}

int pspde_adam_flat(int64_t n, float* theta, const float* grad, float* exp_avg, float* exp_avg_sq, double lr, double beta1,
                    double beta2, double eps, int64_t step, void* stream) {
  if (n < 1 || n > 0x7fffffffLL || !theta || !grad || !exp_avg || !exp_avg_sq || step < 1) return fail(-1, "bad arguments");
  // every scalar is formed in double and rounded once, like the Python floats torch hands to its kernels
  const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
  PSPDE_LAUNCH(adam_flat_kernel, (int)((n + 255) / 256), 256, 0, stream, (int)n, theta, grad, exp_avg, exp_avg_sq,
               (float)(lr / bc1), (float)sqrt(bc2), (float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), (float)eps);
  g_launches++;
  if (const char* e = pspde_peek_error()) return fail(-12, "adam_flat launch failed: %s", e);
  return 0;
}
const char* pspde_last_error(void) { return g_err; }
uint64_t pspde_launch_count(void) { return g_launches.load(); }
void pspde_set_profile_buffer(unsigned long long* dev_buf16) { g_prof = dev_buf16; }

int64_t pspde_theta_size(const pspde_cfg* cfg) {
  // only the network fields matter here (shared by the HJB and the diffusion entry points)
  if (!cfg) { fail(-1, "cfg is NULL"); return -1; }
  if (cfg->n_layers < 1 || cfg->n_layers > PSPDE_MAX_LAYERS || cfg->d < 1 || cfg->time_mode < 0 || cfg->time_mode > 2 ||
      (cfg->net_id != PSPDE_NET_DENSENET && cfg->net_id != PSPDE_NET_MLP_TANH)) { fail(-3, "bad network description"); return -1; }
  NetGeom g;
  if (build_geom(g, cfg->net_id, cfg->n_layers, cfg->dims, cfg->time_mode, cfg->d)) { fail(-3, "bad network geometry"); return -1; }
  return (int64_t)g.n_params * (cfg->time_mode == PSPDE_TIME_NONE ? (cfg->n_sets > 0 ? cfg->n_sets : cfg->N) : 1);
}

size_t pspde_workspace_bytes_fwd(const pspde_cfg* cfg) {
  Plan pl;
  if (make_plan(cfg, false, false, pl)) return 0;
  return pl.stats_bytes + 256;
}

size_t pspde_workspace_bytes(const pspde_cfg* cfg) {
  // upper bound over the entry points that are feasible for cfg (0 if none is)
  Plan pl;
  size_t need = 0;
  if (make_plan(cfg, false, false, pl) == 0) need = pl.stats_bytes;
  if (make_plan(cfg, true, false, pl) == 0) {
    need = pl.stats_bytes + pl.grad_bytes;
#if !defined(PSPDE_EMULATE)
    TcGeom tg;
    CkptPlan cp;
    if (ckpt_plan(cfg, pl, tg, cp)) {
      const size_t n2 = pl.stats_bytes + cp.grad_bytes + cp.ckpt_bytes;
      if (n2 > need) need = n2;
    }
#endif
  }
  if (make_plan(cfg, true, true, pl) == 0) {
    const size_t n3 = pl.stats_bytes + pl.grad_bytes + align256((size_t)pl.grid * cfg->N * kP * cfg->d * sizeof(float));
    if (n3 > need) need = n3;
  }
  return need ? need + 256 : 0;
}

int pspde_rollout_fwd(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0, const float* y0,
                      const float* xi, float* X_N, float* Y_N, float* gX, float* Zsum, double* stats,
                      void* workspace, size_t workspace_bytes, void* stream) {
  return pspde_rollout_fwd_diag(cfg, theta, prob, x0, y0, xi, X_N, Y_N, gX, Zsum, stats, nullptr, workspace,
                                workspace_bytes, stream);
}

int pspde_rollout_fwd_diag(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                           const float* y0, const float* xi, float* X_N, float* Y_N, float* gX, float* Zsum,
                           double* stats, const pspde_udiag* diag, void* workspace, size_t workspace_bytes,
                           void* stream) {
  return pspde_rollout_fwd_ckpt(cfg, theta, prob, x0, y0, xi, X_N, Y_N, gX, Zsum, stats, diag, nullptr, 0, workspace,
                                workspace_bytes, stream);
}

size_t pspde_fwd_ckpt_bytes(const pspde_cfg* cfg) {
  Plan pl;
  if (make_plan(cfg, true, false, pl)) return 0;
  return fwd_ckpt_bytes(cfg, pl);
}

int pspde_rollout_fwd_ckpt(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                           const float* y0, const float* xi, float* X_N, float* Y_N, float* gX, float* Zsum,
                           double* stats, const pspde_udiag* diag, void* ckpt, size_t ckpt_bytes, void* workspace,
                           size_t workspace_bytes, void* stream) {
  Plan pl;
  int rc = make_plan(cfg, false, false, pl);
  if (rc) return rc;
  int keep_tiles = 0;
  if (ckpt) {
    size_t tb = 0;
    const size_t need = fwd_ckpt_bytes(cfg, pl, &tb);
    if (!need) return fail(-6, "configuration is outside the checkpointing forward's shape class");
    if (ckpt_bytes < tb) return fail(-7, "checkpoint buffer too small for one tile (%zu < %zu)", ckpt_bytes, tb);
    keep_tiles = (int)((ckpt_bytes < need ? ckpt_bytes : need) / tb);      // the first tiles that fit
  }
  if (!theta || !prob || !x0) return fail(-1, "theta/prob/x0 must not be NULL");
  if (cfg->noise_mode == PSPDE_NOISE_INJECT && !xi) return fail(-1, "noise_mode INJECT needs xi");
  if (!workspace || workspace_bytes < pl.stats_bytes) return fail(-7, "workspace too small (%zu < %zu)", workspace_bytes, pl.stats_bytes);
  if (misaligned16(workspace)) return fail(-7, "workspace must be 16-byte aligned");
  RolloutParams p;
  fill_params(cfg, pl, p);
  p.theta = theta; p.prob = prob; p.x0 = x0; p.y0 = y0; p.xi = xi;
  p.X_N = X_N; p.Y_N = Y_N; p.gX = gX; p.Zsum = Zsum;
  if (diag && diag->mode != 0) {
    rc = set_udiag(cfg, diag, p);
    if (rc) return rc;
  }
  p.stats_partial = reinterpret_cast<double*>(workspace);
  p.ckpt = reinterpret_cast<float*>(ckpt);
  int grid = pl.grid;
  rc = launch_forward(cfg, pl, p, true, stream, &grid, workspace_bytes, keep_tiles);
  if (rc) return rc;
  if (stats) {
    PSPDE_LAUNCH(reduce_stats_kernel, 1, 32, 0, stream, p.stats_partial, grid, stats);
    g_launches++;
    if (const char* e = pspde_peek_error()) return fail(-12, "reduce_stats launch failed: %s", e);
  }
  return 0;
}

int pspde_rollout_bwd_detached(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                               const float* xi, const float* wY, const float* wZ, float* grad_theta,
                               void* workspace, size_t workspace_bytes, void* stream) {
  Plan pl;
  int rc = make_plan(cfg, true, false, pl);
  if (rc) return rc;
  if (!theta || !prob || !x0 || !wY || !grad_theta) return fail(-1, "theta/prob/x0/wY/grad_theta must not be NULL");
  if (cfg->noise_mode == PSPDE_NOISE_INJECT && !xi) return fail(-1, "noise_mode INJECT needs xi");
  if (!workspace || workspace_bytes < pl.stats_bytes + pl.grad_bytes)
    return fail(-7, "workspace too small (%zu < %zu)", workspace_bytes, pl.stats_bytes + pl.grad_bytes);
  if (misaligned16(workspace)) return fail(-7, "workspace must be 16-byte aligned");
  RolloutParams p;
  fill_params(cfg, pl, p);
  p.theta = theta; p.prob = prob; p.x0 = x0; p.xi = xi; p.wY = wY; p.wZ = wZ;
  p.grad_partial = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + pl.stats_bytes);
#if !defined(PSPDE_EMULATE)
  {
    // Kernel choice (both are this library's CUDA kernels): the checkpointed path -- tensor-core forward that leaves
    // the operand rows of one wave of tiles in the workspace + gradient accumulation kernel -- for the tensor-core
    // shape class when the workspace holds the wave, else the FP32-FMA recompute kernel.  PSPDE_BWD_PATH=simt forces
    // the recompute kernel (A/B tests); PSPDE_BWD_PATH=ckpt makes an ineligible configuration an error.
    TcGeom tg;
    CkptPlan cp;
    const char* path = getenv("PSPDE_BWD_PATH");
    const bool force = path && !strcmp(path, "ckpt");
    bool eligible = ckpt_plan(cfg, pl, tg, cp);
    if (force && !eligible) return fail(-6, "configuration is outside the checkpointed backward's shape class");
    if (eligible && workspace_bytes < pl.stats_bytes + cp.grad_bytes + cp.ckpt_bytes) {
      if (force) return fail(-7, "workspace too small for the checkpointed backward (%zu < %zu)", workspace_bytes,
                             pl.stats_bytes + cp.grad_bytes + cp.ckpt_bytes);
      eligible = false;
    }
    if (eligible && !(path && !strcmp(path, "simt"))) {
      if (pspde_memset0(p.grad_partial, cp.grad_bytes, stream)) return fail(-12, "memset of the gradient partials failed");
      p.ckpt = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + pl.stats_bytes + cp.grad_bytes);
      int used_tc = false;
      rc = run_waves(cfg, pl, p, tg, cp, 0, stream, &used_tc);
      if (rc) return rc;
      return reduce_grad(cfg, pl, p, cp.grid_b, used_tc, grad_theta, stream);
    }
  }
#endif
  if (pspde_memset0(p.grad_partial, (size_t)pl.grid * pl.n_img_total * sizeof(float), stream))
    return fail(-12, "memset of the gradient partials failed");
  if (pl.T == 256) rc = pspde_launch_bwd_256(pl, p, stream);
  else if (pl.T == 512) rc = pspde_launch_bwd_512(pl, p, stream);
  else rc = fail(-13, "internal: no kernel for T=%d NB=%d", pl.T, pl.NB);
  if (rc) return rc;
  return reduce_grad_image(pl, p, pl.grid, grad_theta, stream);
}

int pspde_grad_from_ckpt(const pspde_cfg* cfg, const float* theta, const float* ckpt, int n_slots, int s0,
                         float* grad_theta, void* workspace, size_t workspace_bytes, void* stream) {
  Plan pl;
  int rc = make_plan(cfg, true, false, pl);
  if (rc) return rc;
  if (!theta || !ckpt || !grad_theta || n_slots < 1 || s0 < pl.g.seg_len[0] || (s0 & 7)) return fail(-1, "bad arguments");
  if (pl.g.L != 3 || pl.g.time_mode == TIME_NONE || pl.g.seg_len[1] > 32 || pl.g.seg_len[2] > 32)
    return fail(-6, "configuration is outside the checkpointed backward's shape class");
  const int sms = pspde_sm_count();
  const long long n_ts = (long long)n_slots * cfg->N;
  int grid = n_ts < sms ? (int)n_ts : sms;
  apply_max_grid(grid);
  const size_t gbytes = align256((size_t)grid * grad_part_floats(cfg, pl, s0) * sizeof(float));
  if (!workspace || workspace_bytes < pl.stats_bytes + gbytes) return fail(-7, "workspace too small (%zu < %zu)", workspace_bytes, pl.stats_bytes + gbytes);
  if (misaligned16(workspace)) return fail(-7, "workspace must be 16-byte aligned");
  RolloutParams p;
  fill_params(cfg, pl, p);
  p.theta = theta;
  p.grad_partial = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + pl.stats_bytes);
  p.ckpt = const_cast<float*>(ckpt); p.ckpt_cols = 2 * s0 + 64; p.ckpt_s0 = s0; p.ckpt_zeta = 1;
  if (pspde_memset0(p.grad_partial, gbytes, stream)) return fail(-12, "memset of the gradient partials failed");
  int used_tc = false;
  rc = launch_grad(cfg, pl, p, grid, n_ts, stream, &used_tc);
  if (rc) return rc;
  return reduce_grad(cfg, pl, p, grid, used_tc, grad_theta, stream);
}

int pspde_grad_from_fwd_ckpt(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                             const float* xi, const void* ckpt, size_t ckpt_bytes, const float* wY, float* grad_theta,
                             void* workspace, size_t workspace_bytes, void* stream) {
  Plan pl;
  int rc = make_plan(cfg, true, false, pl);
  if (rc) return rc;
  if (!theta || !ckpt || !wY || !grad_theta) return fail(-1, "theta/ckpt/wY/grad_theta must not be NULL");
#if !defined(PSPDE_EMULATE)
  size_t tb = 0;
  const size_t need = fwd_ckpt_bytes(cfg, pl, &tb);
  if (!need) return fail(-6, "configuration is outside the checkpointing forward's shape class");
  if (ckpt_bytes < tb) return fail(-7, "checkpoint buffer too small for one tile (%zu < %zu)", ckpt_bytes, tb);
  TcGeom tg;
  tc_geom(pl.g, cfg->d, tg);
  const int sms = pspde_sm_count();
  const int n_tiles = (cfg->K_local + kTcP - 1) / kTcP;
  const int n_keep = (int)((ckpt_bytes < need ? ckpt_bytes : need) / tb);       // tiles whose rows the forward kept
  const long long n_ts = (long long)n_keep * cfg->N;
  int grid = n_ts < sms ? (int)n_ts : sms;
  apply_max_grid(grid);
  size_t gbytes = align256((size_t)grid * grad_part_floats(cfg, pl, tg.s0) * sizeof(float));
  size_t ws_need = pl.stats_bytes + gbytes;
  CkptPlan cp;
  if (n_keep < n_tiles) {        // the other tiles: rollout with the cotangents in hand, one wave at a time
    if (!prob || !x0) return fail(-1, "prob/x0 must not be NULL when the buffer does not hold every tile");
    if (cfg->noise_mode == PSPDE_NOISE_INJECT && !xi) return fail(-1, "noise_mode INJECT needs xi");
    TcGeom tg2;
    if (!ckpt_plan(cfg, pl, tg2, cp)) return fail(-6, "configuration is outside the checkpointed backward's shape class");
    if (grid > cp.grid_b) grid = cp.grid_b;
    gbytes = cp.grad_bytes;
    ws_need = pl.stats_bytes + cp.grad_bytes + cp.ckpt_bytes;
  }
  if (!workspace || workspace_bytes < ws_need) return fail(-7, "workspace too small (%zu < %zu)", workspace_bytes, ws_need);
  if (misaligned16(workspace)) return fail(-7, "workspace must be 16-byte aligned");
  RolloutParams p;
  fill_params(cfg, pl, p);
  p.theta = theta; p.prob = prob; p.x0 = x0; p.xi = xi; p.wY = wY;
  p.grad_partial = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + pl.stats_bytes);
  p.ckpt = reinterpret_cast<float*>(const_cast<void*>(ckpt)); p.ckpt_zeta = zeta_in_ckpt(cfg, nullptr);
  p.ckpt_cols = ckpt_cols_of(tg, p.ckpt_zeta); p.ckpt_s0 = tg.s0;
  p.tile0 = 0; p.ckpt_unit = 1;
  if (pspde_memset0(p.grad_partial, gbytes, stream)) return fail(-12, "memset of the gradient partials failed");
  int used_tc = false;
  rc = launch_grad(cfg, pl, p, grid, n_ts, stream, &used_tc);
  if (rc) return rc;
  if (!used_tc) return fail(-13, "internal: the forward checkpoint needs the tensor-core gradient kernel");
  int nparts = grid;
  if (n_keep < n_tiles) {
    p.ckpt = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + pl.stats_bytes + cp.grad_bytes);
    rc = run_waves(cfg, pl, p, tg, cp, n_keep, stream, &used_tc);
    if (rc) return rc;
    nparts = cp.grid_b;
  }
  return reduce_grad(cfg, pl, p, nparts, used_tc, grad_theta, stream);
#else
  (void)prob; (void)x0; (void)xi; (void)ckpt_bytes; (void)workspace; (void)workspace_bytes; (void)stream;
  return fail(-20, "the tensor-core path does not exist in the host emulator");
#endif
}

int pspde_rollout_attached(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                           const float* y0, const float* xi, float w, const float* wY, const float* wZ,
                           const float* wG, float* X_N, float* Y_N, float* gX, float* Zsum, double* stats,
                           float* grad_theta, void* workspace, size_t workspace_bytes, void* stream) {
  return pspde_rollout_attached_diag(cfg, theta, prob, x0, y0, xi, w, wY, wZ, wG, X_N, Y_N, gX, Zsum, stats, nullptr,
                                     grad_theta, workspace, workspace_bytes, stream);
}

int pspde_rollout_attached_diag(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                                const float* y0, const float* xi, float w, const float* wY, const float* wZ,
                                const float* wG, float* X_N, float* Y_N, float* gX, float* Zsum, double* stats,
                                const pspde_udiag* diag, float* grad_theta, void* workspace, size_t workspace_bytes,
                                void* stream) {
  Plan pl;
  int rc = make_plan(cfg, true, true, pl);
  if (rc) return rc;
  if (!cfg->adaptive) return fail(-4, "attached mode implies adaptive_forward_process (solver.py:61-62)");
  if (!theta || !prob || !x0 || !grad_theta) return fail(-1, "theta/prob/x0/grad_theta must not be NULL");
  if (cfg->noise_mode == PSPDE_NOISE_INJECT && !xi) return fail(-1, "noise_mode INJECT needs xi");
  const size_t ckpt_bytes = align256((size_t)pl.grid * cfg->N * kP * cfg->d * sizeof(float));
  if (!workspace || workspace_bytes < pl.stats_bytes + pl.grad_bytes + ckpt_bytes)
    return fail(-7, "workspace too small (%zu < %zu)", workspace_bytes, pl.stats_bytes + pl.grad_bytes + ckpt_bytes);
  if (misaligned16(workspace)) return fail(-7, "workspace must be 16-byte aligned");
  RolloutParams p;
  fill_params(cfg, pl, p);
  p.theta = theta; p.prob = prob; p.x0 = x0; p.y0 = y0; p.xi = xi; p.w_attached = w;
  p.wY = wY; p.wZ = wZ; p.wG = wG;
  p.X_N = X_N; p.Y_N = Y_N; p.gX = gX; p.Zsum = Zsum;
  if (diag && diag->mode != 0) {
    const int rd = set_udiag(cfg, diag, p);
    if (rd) return rd;
  }
  char* ws = reinterpret_cast<char*>(workspace);
  p.stats_partial = reinterpret_cast<double*>(ws);
  p.grad_partial = reinterpret_cast<float*>(ws + pl.stats_bytes);
  p.x_ckpt = reinterpret_cast<float*>(ws + pl.stats_bytes + pl.grad_bytes);
  if (pspde_memset0(p.grad_partial, (size_t)pl.grid * pl.n_img_total * sizeof(float), stream))
    return fail(-12, "memset of the gradient partials failed");
  rc = (pl.T == 256) ? pspde_launch_att_256(pl, p, stream) : pspde_launch_att_512(pl, p, stream);
  if (rc) return rc;
  if (stats) {
    PSPDE_LAUNCH(reduce_stats_kernel, 1, 32, 0, stream, p.stats_partial, pl.grid, stats);
    g_launches++;
  }
  return reduce_grad_image(pl, p, pl.grid, grad_theta, stream);
}

int pspde_importance_sampling(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                              const float* xi, const int32_t* t_index, float dt_net, float* X_N, float* Y_N,
                              float* gX, float* Fint, void* workspace, size_t workspace_bytes, void* stream) {
  Plan pl;
  int rc = make_plan(cfg, false, false, pl);
  if (rc) return rc;
  if (!cfg->adaptive) return fail(-4, "importance sampling simulates the CONTROLLED process (adaptive = 1)");
  if (!theta || !prob || !x0 || !Y_N || !gX || !Fint) return fail(-1, "theta/prob/x0/Y_N/gX/Fint must not be NULL");
  if (cfg->noise_mode == PSPDE_NOISE_INJECT && !xi) return fail(-1, "noise_mode INJECT needs xi");
  if (t_index && !(dt_net > 0.f)) return fail(-2, "dt_net must be > 0 when t_index is given");
  if (!workspace || workspace_bytes < pl.stats_bytes) return fail(-7, "workspace too small");
  if (misaligned16(workspace)) return fail(-7, "workspace must be 16-byte aligned");
  RolloutParams p;
  fill_params(cfg, pl, p);
  p.theta = theta; p.prob = prob; p.x0 = x0; p.xi = xi;
  p.X_N = X_N; p.Y_N = Y_N; p.gX = gX; p.Fint = Fint;
  p.t_index = t_index; p.dt_net = dt_net;
  p.stats_partial = reinterpret_cast<double*>(workspace);
  int grid = pl.grid;
  return launch_forward(cfg, pl, p, true, stream, &grid, workspace_bytes);
}

int pspde_philox_dump(const pspde_cfg* cfg, float* xi_out, void* stream) {
  if (!cfg || !xi_out) return fail(-1, "NULL argument");
  if (cfg->K_local < 1 || cfg->d < 1 || cfg->N < 1) return fail(-2, "bad sizes");
  PSPDE_LAUNCH(philox_dump_kernel, 64, 256, 0, stream, cfg->K_local, cfg->k_offset, cfg->d, cfg->N, cfg->seed,
               cfg->offset, xi_out);
  g_launches++;
  if (const char* e = pspde_peek_error()) return fail(-12, "philox_dump launch failed: %s", e);
  return 0;
}

int64_t pspde_fma_probe(int iters, float* sink, void* stream) { return pspde_fma_probe_ex(0, iters, sink, stream); }

int64_t pspde_fma_probe_ex(int mode, int iters, float* sink, void* stream) {
  const int sms = pspde_sm_count();
  if (sms <= 0 || iters < 1 || !sink || mode < 0 || mode > 2) { fail(-1, "bad arguments"); return -1; }
  if (mode == 0) PSPDE_LAUNCH(fma_probe_kernel<0>, sms, 1024, 0, stream, iters, sink);
  else if (mode == 1) PSPDE_LAUNCH(fma_probe_kernel<1>, sms, 1024, 0, stream, iters, sink);
  else PSPDE_LAUNCH(fma_probe_kernel<2>, sms, 1024, 0, stream, iters, sink);
  g_launches++;
  if (const char* e = pspde_peek_error()) { fail(-12, "fma_probe launch failed: %s", e); return -1; }
  // FLOPs: 16 x 8 FMA-slots per iteration; a packed slot is 2 FMAs, the mixed mode has 4 packed + 8 scalar per 8 slots
  const int64_t fma_per_iter = mode == 0 ? 16 * 8 : mode == 1 ? 16 * 16 : 16 * (4 * 2 + 4 * 2);
  return (int64_t)sms * 1024 * (int64_t)iters * fma_per_iter * 2;
}

}  // extern "C"
