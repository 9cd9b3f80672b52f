// api_common.h -- shared by the api_*.cu translation units: error reporting, validation, launch planning.
#pragma once
#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../include/pspde.h"
#include "rollout_kernels.cuh"

#if defined(PSPDE_EMULATE)
#define PSPDE_LAUNCH(kern, grid, block, smem, stream, ...) \
  emu::launch(dim3(grid), dim3(block), (size_t)(smem), [&]() { kern(__VA_ARGS__); })
static inline int pspde_sm_count() { return emu::M().sm_count; }
static inline int pspde_memset0(void* p, size_t n, void*) { memset(p, 0, n); return 0; }
template <typename K> static inline int pspde_set_smem(K, size_t) { return 0; }
static inline const char* pspde_peek_error() { return nullptr; }
#else
#define PSPDE_LAUNCH(kern, grid, block, smem, stream, ...) \
  kern<<<dim3(grid), dim3(block), (size_t)(smem), (cudaStream_t)(stream)>>>(__VA_ARGS__)
static inline int pspde_sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return -1;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) { n = 0; return -1; }
  }
  return n;
}
static inline int pspde_memset0(void* p, size_t n, void* stream) {
  return cudaMemsetAsync(p, 0, n, (cudaStream_t)stream) == cudaSuccess ? 0 : -1;
}
template <typename K> static inline int pspde_set_smem(K kern, size_t bytes) {
  return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess ? 0 : -1;
}
static inline const char* pspde_peek_error() {
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}
#endif

using namespace pspde;

static_assert(sizeof(pspde_cfg) == 120, "pspde_cfg layout is part of the ABI (mirrored by pspde/_lib.py)");

extern thread_local char g_err[512];
extern std::atomic<unsigned long long> g_launches;
extern unsigned long long* g_prof;   // device buffer for the opt-in phase profiler (pspde_set_profile_buffer)

static inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

constexpr int kP = 64;                       // trajectories per tile
constexpr size_t kMaxSmem = 227 * 1024;      // opt-in dynamic shared memory per CTA on sm_100

struct Plan {
  NetGeom g;
  int T, NB, n_tiles, grid, n_sets, n_theta_total, n_img_total, ctas_per_sm;
  int r_fwd[PSPDE_MAXL];
  size_t smem_bytes, stats_bytes, grad_bytes;
};

static inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }
static inline bool misaligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) != 0; }   // float4 / RED.128 accesses

static inline int validate(const pspde_cfg* c) {
  if (!c) return fail(-1, "cfg is NULL");
  if (c->K_local < 1 || c->d < 1 || c->N < 0) return fail(-2, "bad sizes K_local=%d d=%d N=%d", c->K_local, c->d, c->N);
  if (!(c->dt > 0.f)) return fail(-2, "dt must be > 0");
  if (c->n_layers < 1 || c->n_layers > PSPDE_MAX_LAYERS) return fail(-3, "n_layers=%d unsupported (1..%d)", c->n_layers, PSPDE_MAX_LAYERS);
  if (c->net_id != PSPDE_NET_DENSENET && c->net_id != PSPDE_NET_MLP_TANH) return fail(-3, "unknown net_id %d", c->net_id);
  if (c->time_mode < 0 || c->time_mode > 2) return fail(-3, "unknown time_mode %d", c->time_mode);
  if (c->problem_id != PSPDE_PROBLEM_OU && c->problem_id != PSPDE_PROBLEM_DW)
    return fail(-4, "problem_id %d is not supported by the HJB rollout", c->problem_id);
  if ((c->problem_flags & PSPDE_FLAG_DENSE_AB) && c->d > 128) return fail(-4, "dense A/B needs d <= 128 (d=%d)", c->d);
  if (c->dims[c->n_layers] != c->d) return fail(-3, "control network must map to d outputs (got %d)", c->dims[c->n_layers]);
  if (c->noise_mode != PSPDE_NOISE_INJECT && c->noise_mode != PSPDE_NOISE_PHILOX) return fail(-5, "unknown noise_mode");
  return 0;
}

// rows per thread tile in gemm_nn.  Per k4 step a warp tile of R rows x 4 cols issues 8R FFMA2 (16R FP32-pipe
// cycles on its SMSP) and, as measured with ncu on B200 (profiles/), 4 shared-memory wavefronts per activation
// LDS.128 (8 distinct rows per quarter-warp; quarter-warps do not merge) and 2 per weight LDS.128 (quarter-uniform
// address): 4R + 8 wavefronts at one wavefront per cycle SM wide.  Pick the R that minimises max(pipe time of the
// busiest SMSP, shared-memory time), with a penalty when an SMSP is left with a single warp (nothing to hide the
// LDS latency behind).
static inline int choose_r(int nng, int T, int rmax) {
  const int nw = T / 32;
  int best = 1;
  long best_cost = -1;
  for (int R = 1; R <= rmax; R *= 2) {
    const long nwt = (long)(kP / R / 8) * ((nng + 3) / 4);
    const long waves = (nwt + nw - 1) / nw;
    const long per_wave = nwt < nw ? nwt : nw;
    const long per_smsp = (per_wave + 3) / 4;
    const long pipe = per_smsp * 16 * R, smem = per_wave * (4 * R + 8);
    long cost = waves * (pipe > smem ? pipe : smem);
    if (per_smsp == 1) cost += 40 * waves;
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = R; }
  }
  return best;
}

// Debugging hook PSPDE_MAX_GRID=n: at most n CTAs, so that each CTA loops over more tiles.  make_plan and
// make_diff_plan apply it last, after their own choice of grid (the attached kernel's two CTAs per SM included) and
// before the per-CTA workspace sizes (stats, gradient partials, checkpoints), which follow the grid.  The tensor-core
// launches of api_core.cu (forward, checkpoint rollout, gradient kernels) apply it to their own grids the same way.  A
// workspace sized with the hook set is too small once it is unset: the launch then fails with -7.
static inline void apply_max_grid(int& grid) {
  if (const char* mg = getenv("PSPDE_MAX_GRID")) {
    const int v = atoi(mg);
    if (v > 0 && v < grid) grid = v;
  }
}

static inline int make_plan(const pspde_cfg* c, bool bwd, bool attached, Plan& pl) {
  int rc = validate(c);
  if (rc) return rc;
  rc = build_geom(pl.g, c->net_id, c->n_layers, c->dims, c->time_mode, c->d);
  if (rc) return fail(-3, "network geometry rejected (code %d): dims[0] must be d%s", rc, c->time_mode == PSPDE_TIME_NONE ? "" : "+1");
  pl.n_sets = (c->time_mode == PSPDE_TIME_NONE) ? (c->n_sets > 0 ? c->n_sets : c->N) : 1;
  pl.n_theta_total = pl.g.n_params * pl.n_sets;
  pl.n_img_total = pl.g.w_floats * pl.n_sets;     // one CTA's weight-gradient partial (weight-image layout)
  pl.n_tiles = (c->K_local + kP - 1) / kP;
  const int sms = pspde_sm_count();
  if (sms <= 0) return fail(-10, "no CUDA device");
  pl.grid = pl.n_tiles < sms ? pl.n_tiles : sms;
  pl.T = 512; pl.NB = 1;
  if (bwd) {   // one 8x8 weight-gradient block (64 accumulators) per thread
    const int nb = pl.g.n_blocks;
    if (nb <= 224) pl.T = 256;           // leaves a spare warp for the row-split leftover blocks
    else if (nb <= 512) pl.T = 512;
    else return fail(-6, "network too large for the register-resident gradient path (%d 8x8 blocks > 512)", nb);
  }
  for (int l = 0; l < pl.g.L; ++l) pl.r_fwd[l] = choose_r(pl.g.layer[l].nng, pl.T, bwd ? 4 : 8);
  const SmemLayout sl = smem_layout(pl.g, kP, bwd, attached);
  pl.smem_bytes = (size_t)sl.total * sizeof(float);
  if (pl.smem_bytes > kMaxSmem)
    return fail(-6, "network + tile need %zu B of shared memory (> %zu)", pl.smem_bytes, kMaxSmem);
  // Attached kernel, 256 threads: alone on an SM it runs at 208 registers with 8 warps (ncu: FMA pipe 24 %, warps stalled on
  // fixed latencies, profiles/r02_attached_ncu_full_summary.json).  Two CTAs per SM at <= 128 registers (75 spilled floats)
  // are 31 % faster at the C3 shape (205 -> 156 ms), so that is the default whenever two tiles' shared memory fits;
  // PSPDE_ATT_CTAS=1 restores one CTA per SM.
  pl.ctas_per_sm = 1;
  if (attached && pl.T == 256 && 2 * (pl.smem_bytes + 1024) <= kMaxSmem + 1024) {
    const char* e = getenv("PSPDE_ATT_CTAS");
    if (!(e && e[0] == '1')) { pl.ctas_per_sm = 2; pl.grid = pl.n_tiles < 2 * sms ? pl.n_tiles : 2 * sms; }
  }
  apply_max_grid(pl.grid);
  pl.stats_bytes = align256((size_t)pl.grid * 4 * sizeof(double));
  pl.grad_bytes = bwd ? align256((size_t)pl.grid * pl.n_img_total * sizeof(float)) : 0;
  return 0;
}

const int* pspde_theta_table(const pspde::NetGeom& g);   // api_core.cu

static inline void fill_params(const pspde_cfg* c, const Plan& pl, RolloutParams& p) {
  memset(&p, 0, sizeof(p));
  p.g = pl.g;
  p.K_local = c->K_local; p.k_offset = c->k_offset; p.d = c->d; p.N = c->N; p.dt = c->dt;
  p.problem_id = c->problem_id; p.flags = c->problem_flags; p.adaptive = c->adaptive;
  p.noise_mode = c->noise_mode; p.x0_per_path = c->x0_per_path;
  p.seed = c->seed; p.offset = c->offset;
  p.xs_k = c->xi_stride_k; p.xs_j = c->xi_stride_j; p.xs_n = c->xi_stride_n;
  p.n_tiles = pl.n_tiles; p.n_theta_total = pl.n_theta_total; p.n_img_total = pl.n_img_total;
  for (int l = 0; l < PSPDE_MAXL; ++l) p.r_fwd[l] = pl.r_fwd[l];
  p.prof = g_prof;
  p.n_sets = pl.n_sets;
  p.u_quirk = -1;
  p.d_abs_max = c->d_abs_max > 0.f ? c->d_abs_max : INFINITY;
  p.th_tbl = pspde_theta_table(pl.g);   // nullptr = allocation failure: the launchers of the gradient kernels report it
}

template <int T, bool BWD, int NB>
static inline int launch_rollout(const Plan& pl, const RolloutParams& p, void* stream) {
  if (BWD && !p.th_tbl) return fail(-13, "could not allocate the weight-image index table");
  auto kern = rollout_kernel<kP, T, BWD, NB>;
  if (pspde_set_smem(kern, pl.smem_bytes)) return fail(-11, "cudaFuncSetAttribute(%zu B smem) failed", pl.smem_bytes);
  PSPDE_LAUNCH(kern, pl.grid, T, pl.smem_bytes, stream, p);
  g_launches++;
  if (const char* e = pspde_peek_error()) return fail(-12, "rollout kernel launch failed: %s", e);
  return 0;
}



// gradient accumulation from the checkpoint buffer (grad_kernels.cuh); grid CTAs, n_items work items
int pspde_launch_grad_256(const Plan& pl, const pspde::RolloutParams& p, int grid, int n_items, void* stream);
int pspde_launch_grad_512(const Plan& pl, const pspde::RolloutParams& p, int grid, int n_items, void* stream);

// defined in api_bwd*.cu / api_att*.cu (one translation unit per thread count so that the template instantiations
// compile in parallel)
int pspde_launch_bwd_256(const Plan& pl, const pspde::RolloutParams& p, void* stream);
int pspde_launch_bwd_512(const Plan& pl, const pspde::RolloutParams& p, void* stream);
int pspde_launch_att_256(const Plan& pl, const pspde::RolloutParams& p, void* stream);
int pspde_launch_att_512(const Plan& pl, const pspde::RolloutParams& p, void* stream);
