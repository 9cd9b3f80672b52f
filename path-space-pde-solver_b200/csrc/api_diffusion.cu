// api_diffusion.cu -- extern "C" entry points of the diffusion-loss rollout (GeneralSolver, solver.py:1076-1163, and
// its elliptic sibling EllipticSolver, solver.py:628-790).
#include "api_common.h"
#include "diffusion_kernels.cuh"

namespace {

constexpr int kPD = 32;      // paths per tile (2 * kPD rows: value + tangent)
constexpr int kTD = 512;

struct DiffPlan {
  NetGeom g;
  int n_tiles, grid;
  size_t smem_bytes, stats_bytes, wpack_bytes, grad_bytes;
};

int validate_diffusion(const pspde_cfg* c, float T_end, const pspde_elliptic* ell = nullptr) {
  if (!c) return fail(-1, "cfg is NULL");
  if (c->K_local < 1 || c->d < 1 || c->N < 0) return fail(-2, "bad sizes K_local=%d d=%d N=%d", c->K_local, c->d, c->N);
  if (!(c->dt > 0.f) || !(T_end > 0.f)) return fail(-2, "dt and T must be > 0");
  if (ell) {
    if (c->n_layers < 1 || c->n_layers > PSPDE_MAX_LAYERS) return fail(-3, "n_layers=%d unsupported (1..%d)", c->n_layers, PSPDE_MAX_LAYERS);
    if (c->net_id != PSPDE_NET_DENSENET) return fail(-3, "the diffusion loss needs a DenseNet value function (function_space.py:116-140)");
    if (c->time_mode != PSPDE_TIME_NONE) return fail(-3, "the elliptic value network sees X only (solver.py:606): time_mode must be TIME_NONE");
    if (c->dims[c->n_layers] != 1) return fail(-3, "the value network has one output (got %d)", c->dims[c->n_layers]);
    if (c->problem_id != PSPDE_PROBLEM_HEAT && c->problem_id != PSPDE_PROBLEM_OU)
      return fail(-4, "problem_id %d is not supported by the diffusion rollout (drift a_diag x, diffusion diag(b_diag))", c->problem_id);
    if (c->problem_flags & PSPDE_FLAG_DENSE_AB) return fail(-4, "the diffusion rollout needs diagonal drift / diffusion");
    if (c->noise_mode != PSPDE_NOISE_INJECT && c->noise_mode != PSPDE_NOISE_PHILOX) return fail(-5, "unknown noise_mode");
    if (ell->domain == PSPDE_DOMAIN_SPHERE) { if (!(ell->radius > 0.f)) return fail(-2, "sphere radius must be > 0"); }
    else if (ell->domain == PSPDE_DOMAIN_BOX) { if (!(ell->x_r > ell->x_l)) return fail(-2, "box needs x_l < x_r"); }
    else if (ell->domain == PSPDE_DOMAIN_ANNULUS) { if (!(ell->radius > ell->radius_in) || !(ell->radius_in > 0.f)) return fail(-2, "annulus needs 0 < radius_in < radius"); }
    else return fail(-4, "unknown domain %d (PSPDE_DOMAIN_SPHERE | PSPDE_DOMAIN_BOX | PSPDE_DOMAIN_ANNULUS)", ell->domain);
    if (!(ell->h_id >= PSPDE_H_ZERO && ell->h_id <= PSPDE_H_HELMHOLTZ) && ell->h_id != PSPDE_H_COMMITTOR) return fail(-4, "unknown h_id %d", ell->h_id);
    if (ell->h_id == PSPDE_H_HELMHOLTZ && c->d < 2) return fail(-4, "the Helmholtz right-hand side needs d >= 2 (problems.py:1628)");
    return 0;
  }
  if (c->n_layers < 1 || c->n_layers > PSPDE_MAX_LAYERS) return fail(-3, "n_layers=%d unsupported (1..%d)", c->n_layers, PSPDE_MAX_LAYERS);
  if (c->net_id != PSPDE_NET_DENSENET) return fail(-3, "the diffusion loss needs a DenseNet value function (function_space.py:116-140)");
  if (c->time_mode != PSPDE_TIME_LAST) return fail(-3, "the value network sees [X, t] (solver.py:1079): time_mode must be TIME_LAST");
  if (c->dims[c->n_layers] != 1) return fail(-3, "the value network has one output (got %d)", c->dims[c->n_layers]);
  if (c->problem_id != PSPDE_PROBLEM_HEAT && c->problem_id != PSPDE_PROBLEM_OU && c->problem_id != PSPDE_PROBLEM_ALLEN_CAHN)
    return fail(-4, "problem_id %d is not supported by the diffusion rollout (h = 0 or Allen-Cahn)", c->problem_id);
  if (c->problem_flags & PSPDE_FLAG_DENSE_AB) return fail(-4, "the diffusion rollout needs diagonal drift / diffusion");
  if (c->noise_mode != PSPDE_NOISE_INJECT && c->noise_mode != PSPDE_NOISE_PHILOX) return fail(-5, "unknown noise_mode");
  return 0;
}

int make_diff_plan(const pspde_cfg* c, float T_end, DiffPlan& pl, const pspde_elliptic* ell = nullptr) {
  int rc = validate_diffusion(c, T_end, ell);
  if (rc) return rc;
  rc = build_geom(pl.g, c->net_id, c->n_layers, c->dims, c->time_mode, c->d);
  if (rc) return fail(-3, "network geometry rejected (code %d): dims[0] must be %s", rc, ell ? "d" : "d+1");
  pl.n_tiles = (c->K_local + kPD - 1) / kPD;
  const int sms = pspde_sm_count();
  if (sms <= 0) return fail(-10, "no CUDA device");
  pl.grid = pl.n_tiles < sms ? pl.n_tiles : sms;
  pl.smem_bytes = (size_t)diff_smem_layout(pl.g, kPD).total * sizeof(float);
  if (pl.smem_bytes > kMaxSmem) return fail(-6, "network + tile need %zu B of shared memory (> %zu)", pl.smem_bytes, kMaxSmem);
  apply_max_grid(pl.grid);
  pl.stats_bytes = align256((size_t)pl.grid * 4 * sizeof(double));
  pl.wpack_bytes = align256((size_t)pl.g.w_floats * sizeof(float));
  pl.grad_bytes = align256((size_t)pl.grid * dw_partial_floats(pl.g) * sizeof(float));
  return 0;
}

void fill_diff_params(const pspde_cfg* c, float T_end, const DiffPlan& pl, DiffusionParams& p) {
  memset(&p, 0, sizeof(p));
  p.g = pl.g;
  p.K_local = c->K_local; p.k_offset = c->k_offset; p.d = c->d; p.N = c->N; p.dt = c->dt; p.T_end = T_end;
  p.noise_mode = c->noise_mode; p.seed = c->seed; p.offset = c->offset;
  p.xs_n = c->xi_stride_n; p.xs_k = c->xi_stride_k; p.xs_j = c->xi_stride_j;
  p.n_tiles = pl.n_tiles;
  if (c->problem_id == PSPDE_PROBLEM_ALLEN_CAHN) { p.hf.id = HFUN_ALLEN_CAHN; p.hf.d = c->d; }     // h = y - y^3 (problems.py:1203)
}

void fill_elliptic(const pspde_cfg* c, const pspde_elliptic* ell, DiffusionParams& p) {
  p.domain = ell->domain == PSPDE_DOMAIN_SPHERE ? DOMAIN_SPHERE : ell->domain == PSPDE_DOMAIN_BOX ? DOMAIN_BOX : DOMAIN_ANNULUS;
  p.radius = ell->radius; p.x_l = ell->x_l; p.x_r = ell->x_r; p.one_boundary = ell->one_boundary; p.radius_in = ell->radius_in;
  p.hf.id = ell->h_id; p.hf.d = c->d; p.hf.p0 = ell->h_param[0]; p.hf.p1 = ell->h_param[1]; p.hf.p2 = ell->h_param[2];
}

int pack_weights(const DiffPlan& pl, const float* theta, float* wpack, void* stream) {
  PSPDE_LAUNCH(pack_weights_kernel, 64, 256, 0, stream, pl.g, theta, wpack);
  g_launches++;
  if (const char* e = pspde_peek_error()) return fail(-12, "pack_weights launch failed: %s", e);
  return 0;
}

template <bool BWD>
int launch_diffusion(const DiffPlan& pl, const DiffusionParams& p, void* stream) {
  auto kern = diffusion_kernel<kPD, kTD, BWD>;
  if (pspde_set_smem(kern, pl.smem_bytes)) return fail(-11, "cudaFuncSetAttribute(%zu B smem) failed", pl.smem_bytes);
  PSPDE_LAUNCH(kern, pl.grid, kTD, pl.smem_bytes, stream, p);
  g_launches++;
  if (const char* e = pspde_peek_error()) return fail(-12, "diffusion kernel launch failed: %s", e);
  return 0;
}

}  // namespace

extern "C" {

size_t pspde_diffusion_workspace_bytes(const pspde_cfg* cfg, float T_end) {
  DiffPlan pl;
  if (make_diff_plan(cfg, T_end, pl)) return 0;
  return pl.stats_bytes + pl.wpack_bytes + pl.grad_bytes + 256;
}

static int diffusion_fwd_impl(const pspde_cfg* cfg, float T_end, const pspde_elliptic* ell, const float* theta,
                              const float* prob, const float* X0, const float* t0, const float* xi, float* V0,
                              float* VE, float* Y_end, float* X_end, float* t_end, float* VL2, double* stats,
                              void* workspace, size_t workspace_bytes, void* stream) {
  DiffPlan pl;
  int rc = make_diff_plan(cfg, T_end, pl, ell);
  if (rc) return rc;
  if (!theta || !prob || !X0 || (!ell && !t0)) return fail(-1, "theta/prob/X0/t0 must not be NULL");
  if (cfg->noise_mode == PSPDE_NOISE_INJECT && cfg->N > 0 && !xi) return fail(-1, "noise_mode INJECT needs xi");
  if (!workspace || workspace_bytes < pl.stats_bytes + pl.wpack_bytes)
    return fail(-7, "workspace too small (%zu < %zu)", workspace_bytes, pl.stats_bytes + pl.wpack_bytes);
  if (misaligned16(workspace)) return fail(-7, "workspace must be 16-byte aligned");
  char* ws = reinterpret_cast<char*>(workspace);
  float* wpack = reinterpret_cast<float*>(ws + pl.stats_bytes);
  rc = pack_weights(pl, theta, wpack, stream);
  if (rc) return rc;
  DiffusionParams p;
  fill_diff_params(cfg, T_end, pl, p);
  p.wpack = wpack; p.prob = prob; p.X0 = X0; p.t0 = t0; p.xi = xi;
  p.V0 = V0; p.VE = VE; p.Y_end = Y_end; p.X_end = X_end; p.t_end = t_end; p.VL2 = VL2;
  if (ell) fill_elliptic(cfg, ell, p);
  p.stats_partial = reinterpret_cast<double*>(ws);
  rc = launch_diffusion<false>(pl, p, stream);
  if (rc) return rc;
  if (stats) {
    PSPDE_LAUNCH(reduce_stats_kernel, 1, 32, 0, stream, p.stats_partial, pl.grid, 1, stats);
    g_launches++;
    if (const char* e = pspde_peek_error()) return fail(-12, "reduce_stats launch failed: %s", e);
  }
  return 0;
}

static int diffusion_bwd_impl(const pspde_cfg* cfg, float T_end, const pspde_elliptic* ell, const float* theta,
                              const float* prob, const float* X0, const float* t0, const float* xi, const float* c0,
                              const float* cE, const float* cD, float* grad_theta, void* workspace,
                              size_t workspace_bytes, void* stream) {
  DiffPlan pl;
  int rc = make_diff_plan(cfg, T_end, pl, ell);
  if (rc) return rc;
  if (!theta || !prob || !X0 || (!ell && !t0) || !grad_theta) return fail(-1, "theta/prob/X0/t0/grad_theta must not be NULL");
  if (cfg->noise_mode == PSPDE_NOISE_INJECT && cfg->N > 0 && !xi) return fail(-1, "noise_mode INJECT needs xi");
  const size_t need = pl.stats_bytes + pl.wpack_bytes + pl.grad_bytes;
  if (!workspace || workspace_bytes < need) return fail(-7, "workspace too small (%zu < %zu)", workspace_bytes, need);
  if (misaligned16(workspace)) return fail(-7, "workspace must be 16-byte aligned");
  char* ws = reinterpret_cast<char*>(workspace);
  float* wpack = reinterpret_cast<float*>(ws + pl.stats_bytes);
  rc = pack_weights(pl, theta, wpack, stream);
  if (rc) return rc;
  DiffusionParams p;
  fill_diff_params(cfg, T_end, pl, p);
  p.wpack = wpack; p.prob = prob; p.X0 = X0; p.t0 = t0; p.xi = xi;
  p.c0 = c0; p.cE = cE; p.cD = cD;
  if (ell) fill_elliptic(cfg, ell, p);
  p.grad_partial = reinterpret_cast<float*>(ws + pl.stats_bytes + pl.wpack_bytes);
  if (pspde_memset0(p.grad_partial, (size_t)pl.grid * dw_partial_floats(pl.g) * sizeof(float), stream))
    return fail(-12, "memset of the gradient partials failed");
  rc = launch_diffusion<true>(pl, p, stream);
  if (rc) return rc;
  const int tot = pl.g.n_blocks * 64;
  PSPDE_LAUNCH(reduce_dw_kernel, (tot + 255) / 256, 256, 0, stream, pl.g, p.grad_partial, pl.grid, grad_theta);
  g_launches++;
  if (const char* e = pspde_peek_error()) return fail(-12, "reduce_dw launch failed: %s", e);
  return 0;
}

int pspde_diffusion_fwd(const pspde_cfg* cfg, float T_end, const float* theta, const float* prob, const float* X0,
                        const float* t0, const float* xi, float* V0, float* VE, float* Y_end, float* X_end,
                        float* t_end, double* stats, void* workspace, size_t workspace_bytes, void* stream) {
  return diffusion_fwd_impl(cfg, T_end, nullptr, theta, prob, X0, t0, xi, V0, VE, Y_end, X_end, t_end, nullptr, stats,
                            workspace, workspace_bytes, stream);
}

int pspde_diffusion_bwd(const pspde_cfg* cfg, float T_end, const float* theta, const float* prob, const float* X0,
                        const float* t0, const float* xi, const float* c0, const float* cE, const float* cD,
                        float* grad_theta, void* workspace, size_t workspace_bytes, void* stream) {
  return diffusion_bwd_impl(cfg, T_end, nullptr, theta, prob, X0, t0, xi, c0, cE, cD, grad_theta, workspace,
                            workspace_bytes, stream);
}

size_t pspde_elliptic_workspace_bytes(const pspde_cfg* cfg, const pspde_elliptic* ell) {
  DiffPlan pl;
  if (!ell) { fail(-1, "ell is NULL"); return 0; }
  if (make_diff_plan(cfg, 1.0f, pl, ell)) return 0;
  return pl.stats_bytes + pl.wpack_bytes + pl.grad_bytes + 256;
}

int pspde_elliptic_fwd(const pspde_cfg* cfg, const pspde_elliptic* ell, const float* theta, const float* prob,
                       const float* X0, const float* xi, float* V0, float* VE, float* Y_end, float* X_end,
                       float* VL2, double* stats, void* workspace, size_t workspace_bytes, void* stream) {
  if (!ell) return fail(-1, "ell is NULL");
  return diffusion_fwd_impl(cfg, 1.0f, ell, theta, prob, X0, nullptr, xi, V0, VE, Y_end, X_end, nullptr, VL2, stats,
                            workspace, workspace_bytes, stream);
}

int pspde_elliptic_bwd(const pspde_cfg* cfg, const pspde_elliptic* ell, const float* theta, const float* prob,
                       const float* X0, const float* xi, const float* c0, const float* cE, const float* cD,
                       float* grad_theta, void* workspace, size_t workspace_bytes, void* stream) {
  if (!ell) return fail(-1, "ell is NULL");
  return diffusion_bwd_impl(cfg, 1.0f, ell, theta, prob, X0, nullptr, xi, c0, cE, cD, grad_theta, workspace,
                            workspace_bytes, stream);
}

int pspde_diffusion_sample(const pspde_cfg* cfg, float radius, float T_end, float* X0, float* t0, void* stream) {
  if (!cfg || !X0 || !t0) return fail(-1, "NULL argument");
  if (cfg->K_local < 1 || cfg->d < 1 || !(radius > 0.f) || !(T_end > 0.f)) return fail(-2, "bad sizes");
  const int sms = pspde_sm_count();
  if (sms <= 0) return fail(-10, "no CUDA device");
  PSPDE_LAUNCH(diffusion_sample_kernel, 2 * sms, 256, 0, stream, cfg->K_local, cfg->k_offset, cfg->d, radius, T_end,
               cfg->seed, cfg->offset, X0, t0);
  g_launches++;
  if (const char* e = pspde_peek_error()) return fail(-12, "diffusion_sample launch failed: %s", e);
  return 0;
}

}  // extern "C"
