/* pspde.h -- C ABI of libpspde: the B200 (sm_100a) fused path-space rollout.
 *
 * The reference (lorenzrichter/path-space-PDE-solver) has no FFI; its de-facto boundary for the hot path is
 * the body of Solver.train (solver.py:433-499: initialize_training_data -> N-step Euler-Maruyama loop ->
 * loss_function -> loss.backward) and of GeneralSolver.train (solver.py:1040-1188).  Each entry point below
 * replaces one slice of that body; the reference lines it stands for are cited at the declaration.
 *
 * Conventions
 *   - plain C, plain pointers and sizes; no torch types.  All buffer arguments of the device entry points
 *     are DEVICE pointers owned by the caller.  `workspace` and `ckpt` buffers must be at least 16-byte aligned (checked; cudaMalloc
 *     and the torch allocator return 256 / 512): the kernels address them with 16-byte vector accesses and TMA.  The library keeps only
 *     two small caches of its own on the device (a packed weight image per stream that launched a tensor-core rollout, an
 *     index table per network geometry; INTEGRATION.md, "Ownership").
 *   - every call only enqueues work on `stream` (a cudaStream_t passed as void*); no host synchronisation,
 *     re-entrant per device, one process per GPU.  The *_host entry point is the exception (documented there).
 *   - return value 0 = ok; negative = error, message via pspde_last_error() (thread local).  Never throws.
 *   - fp32 arithmetic throughout (dtype "f32"); loss statistics are accumulated in fp64.
 */
#ifndef PSPDE_H
#define PSPDE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSPDE_ABI_VERSION 3
#define PSPDE_MAX_LAYERS 4          /* linear layers per network (<= 3 hidden) */

/* problem functors (problems.py): drift b(x), diffusion sigma = B, running cost f, terminal cost g.
 *   PSPDE_PROBLEM_OU   LLGC (problems.py:14-49) and LQGC (:118-167):
 *                      b = A x, sigma = B, f = x'Px, g = alpha.x + x'Rx, h = -|z|^2/2 - f
 *   PSPDE_PROBLEM_DW   DoubleWell(_multidim) (problems.py:178-214, :285-334):
 *                      b_i = -4 kappa_i x_i (x_i^2 - 1), sigma = I, f = 0, g = sum eta_i (x_i - 1)^2
 *   PSPDE_PROBLEM_HEAT HeatEquation (problems.py:1733-1764), diffusion loss only:
 *                      b = 0, sigma = sqrt(2) I, h = 0, terminal f = |x|^2
 *   PSPDE_PROBLEM_ALLEN_CAHN AllenCahn (problems.py:1175-1218), diffusion loss only:
 *                      b = 0, sigma = sqrt(2) I, h = y - y^3, terminal f = 1 / (2 + 2/5 |x|^2)
 * Parameter pack `prob` (fp32): 7 vectors of length d, in this order
 *      a_diag | b_diag | p_diag | r_diag | alpha | kappa | eta
 * followed, when PSPDE_FLAG_DENSE_AB is set, by the row-major d x d matrices A then B (the diagonal
 * vectors are then ignored for drift/diffusion).  P and R are diagonal in every reference problem. */
enum { PSPDE_PROBLEM_OU = 0, PSPDE_PROBLEM_DW = 1, PSPDE_PROBLEM_HEAT = 2, PSPDE_PROBLEM_ALLEN_CAHN = 3 };
enum { PSPDE_FLAG_DENSE_AB = 1 };

/* networks (function_space.py).  theta is the flat concatenation of module.parameters():
 *   PSPDE_NET_DENSENET  DenseNet (:116-140): W_i (sum(dims[:i+1]), dims[i+1]) row major, b_i; act relu(.)^2
 *   PSPDE_NET_MLP_TANH  MySequential (:177-195): nn.Linear weight_i (dims[i+1], dims[i]), bias_i; act tanh */
enum { PSPDE_NET_DENSENET = 0, PSPDE_NET_MLP_TANH = 1 };

/* where time enters the network input (solver.py:349-356, :1079):
 *   TIME_FIRST  'inner': input [t_n, X]            (Solver)
 *   TIME_NONE   'outer': input X, one parameter set per step, theta = N stacked sets
 *   TIME_LAST   input [X, t]                       (GeneralSolver) */
enum { PSPDE_TIME_FIRST = 0, PSPDE_TIME_NONE = 1, PSPDE_TIME_LAST = 2 };

/* Brownian increments: INJECT reads xi from memory (parity with solver.py:381), PHILOX generates them in
 * the kernel: Philox4x32-10, counter (k_global, n, j/4, offset), key = seed, Box-Muller. */
enum { PSPDE_NOISE_INJECT = 0, PSPDE_NOISE_PHILOX = 1 };

typedef struct pspde_cfg {
  int32_t K_local;      /* trajectories simulated by this call (this GPU's shard)                  */
  int32_t k_offset;     /* global index of the first local trajectory (Philox counter)             */
  int32_t d;            /* state dimension                                                         */
  int32_t N;            /* Euler-Maruyama steps (computed on the host: solver.py:41)               */
  float   dt;           /* step size as fp32 (solver.py:39); sqrt(dt) is taken in fp32 (:40)       */
  int32_t problem_id;   /* PSPDE_PROBLEM_*                                                         */
  int32_t problem_flags;
  int32_t net_id;       /* PSPDE_NET_*                                                             */
  int32_t n_layers;     /* number of linear layers L (dims has L+1 entries)                        */
  int32_t dims[PSPDE_MAX_LAYERS + 1];  /* [d_in, h_1, ..., d_out]; d_in includes the time column   */
  int32_t time_mode;    /* PSPDE_TIME_*                                                            */
  int32_t adaptive;     /* adaptive_forward_process: c = -Z (solver.py:452-456) else c = 0         */
  int32_t noise_mode;   /* PSPDE_NOISE_*                                                           */
  int32_t x0_per_path;  /* 0: x0 is one row of d floats (X_0.repeat, :365); 1: K_local x d rows    */
  uint64_t seed;        /* Philox key                                                              */
  uint32_t offset;      /* Philox stream id: the training-iteration counter                       */
  int32_t  n_sets;      /* TIME_NONE: number of stacked parameter sets in theta (0 = N)            */
  /* INJECT: element (k, j, step n) is read at xi[k*xi_stride_k + j*xi_stride_j + n*xi_stride_n], n = 0..N-1
   * being the increment that drives step n.  Reference layout (K, d, N+1) with slice n+1 driving step n
   * (solver.py:472): pass xi + 1 and strides (d*(N+1), N+1, 1). */
  int64_t xi_stride_k, xi_stride_j, xi_stride_n;
  /* Blow-up bound: a trajectory whose |D| = |Y_N - g(X_N)| reaches d_abs_max is dropped from the batch exactly like one
   * with a non-finite D (counted in stats[3], Y_N written as NaN, zero cotangent).  The untrained relu(.)^2 feedback
   * control drives about one path in 10^5 to |D| ~ 10^20 .. 10^30 -- finite, but one such value makes the log-variance
   * loss 10^34 and its gradient inf (the reference returns NaN for the whole batch from then on).  0 = off. */
  float   d_abs_max;
} pspde_cfg;

int          pspde_abi_version(void);
const char*  pspde_last_error(void);
/* number of kernels launched by this library in this process so far (bench.py's gpu_launches) */
uint64_t     pspde_launch_count(void);
/* Debug hook: when set to a device buffer of 32 uint64 (zeroed by the caller), CTA 0 of the detached rollout
 * kernels adds clock64() cycles per phase: [0] step prologue, [1] network forward, [2] SDE step, [3] hidden
 * cotangents, [4] weight gradient.  NULL (default) disables it. */
void         pspde_set_profile_buffer(unsigned long long* dev_buf16);
/* number of parameters in theta for cfg (all N sets in TIME_NONE mode); <0 on invalid cfg */
int64_t      pspde_theta_size(const pspde_cfg* cfg);
/* scratch bytes the rollout entry points need for cfg (upper bound over all of them; for the tensor-core shape
 * class this includes the per-wave checkpoint buffer of pspde_rollout_bwd_detached, <= 24 GB) */
size_t       pspde_workspace_bytes(const pspde_cfg* cfg);
/* scratch bytes of the forward-only entry points (pspde_rollout_fwd / _fwd_diag, pspde_importance_sampling) */
size_t       pspde_workspace_bytes_fwd(const pspde_cfg* cfg);

/* Forward rollout -- replaces solver.py:433-494 (initialize_training_data + the N-step loop) and the
 * reductions of loss_function (:164-192).  Per path: X_N (nullable, K x d), Y_N, gX = g(X_N),
 * Zsum = sum_n (|Z|^2/2 + f(X_{n+1})) dt (:486).  y0 (nullable) is a device scalar added to Y (learn_Y_0, :372-373).
 * stats (nullable) receives 4 doubles: sum D, sum D^2 (D = Y_N - gX), sum (Zsum + gX), #non-finite D. */
int pspde_rollout_fwd(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                      const float* y0, const float* xi, float* X_N, float* Y_N, float* gX, float* Zsum,
                      double* stats, void* workspace, size_t workspace_bytes, void* stream);

/* u_L2 diagnostic of solver.py:491-494, u_L2 += sum_j (-Z_j - u*_j(X_{n+1}, n*delta_t))^2 dt, evaluated in the
 * forward kernel from per-step device tables instead of the reference's per-step D2H / scipy / H2D round trip:
 *   mode 1  u*_j = U0[n][j] + U1[n][j] * x_j          table fp32 [N][2][d]   (LLGC problems.py:51-53: U1 = 0;
 *                                                      LQGC :169-171 with diagonal Q^-1 B' F_n: U0 = 0)
 *   mode 2  u*_j = tab[n][j < d1 ? 0 : 1][cell(x_j)]  table fp32 [N][2][nx1], cell = floor((clip(x, -xb, xb - 2dx) + xb) / dx)
 *                                                      (DoubleWell(_multidim) finite-difference tables, :398-404, :463-476)
 *           quirk_path >= 0: the path with that GLOBAL index reads its cell two to the left, a negative cell wrapping to the
 *           table's end -- the reference's `i[-1] -= 2` on the last batch element (problems.py:279, :401, :464) followed by
 *           numpy's negative indexing; -1 switches it off */
typedef struct pspde_udiag {
  int32_t mode;          /* 0 off */
  int32_t nx1, d1;       /* mode 2 */
  float   xb, dx;        /* mode 2 */
  const float* table;    /* device */
  float*  uL2;           /* device, K_local per-path results */
  int32_t quirk_path;    /* mode 2: global path index of the `i[-1] -= 2` element, or -1 */
} pspde_udiag;

int pspde_rollout_fwd_diag(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                           const float* y0, const float* xi, float* X_N, float* Y_N, float* gX, float* Zsum,
                           double* stats, const pspde_udiag* diag, void* workspace, size_t workspace_bytes,
                           void* stream);

/* Backward for detach_forward=True (solver.py:468-469 + loss.backward at :221).  The trajectories do not
 * depend on theta, so dLoss/dtheta = sum_{k,n} J_theta Z(t_n, X_{k,n})' zeta_{k,n} with
 *   zeta = wY_k (sqrt(dt) xi_{n+1} + [adaptive == 0] Z dt) + wZ_k Z dt,
 * wY = dLoss/dY_N, wZ = dLoss/dZsum (nullable = 0), both of length K_local.  The rollout is recomputed
 * from (x0, xi | Philox); this entry point keeps nothing of size K x N x d in HBM (its checkpoint buffer holds one wave
 * of tiles, independent of K; the opt-in K-proportional row buffer belongs to pspde_rollout_fwd_ckpt below).
 * grad_theta (pspde_theta_size floats) is overwritten.
 * Two kernel families implement it: for the tensor-core shape class (see DESIGN.md) the trajectories of one wave of
 * tiles (<= one 128-path tile per SM) are regenerated by the tensor-core forward kernel, which checkpoints the
 * per-step operand rows in the workspace, and a gradient kernel streams them back (pspde_grad_from_ckpt); any other
 * configuration, or a workspace smaller than pspde_workspace_bytes(), runs the FP32-FMA recompute kernel. */
int pspde_rollout_bwd_detached(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                               const float* xi, const float* wY, const float* wZ, float* grad_theta,
                               void* workspace, size_t workspace_bytes, void* stream);

/* Second half of the checkpointed detached backward, exposed for tests: accumulates dLoss/dtheta from the operand
 * rows [a0 | h1 | h2 | zeta] of n_slots tiles of 128 paths x cfg->N steps.  Layout of ckpt (device, fp32): COLUMN-major
 * with the 128 paths of a tile contiguous (one 512-byte row per column: the K-major operand form, K = sample, that the
 * tensor-core gradient kernel loads by TMA),
 *     ckpt[((slot * N + n) * C + col) * 128 + path],   C = 2 * s0 + 64,
 * columns [0, s0) = a0 = [X_n | t_n | 1 | 0..], then 32 columns h1, 32 columns h2 (hidden widths padded to 32, with the
 * constant-1 column of MySequential), then s0 columns zeta (d used); s0 = the input segment padded to a multiple
 * of 8.  pspde_rollout_bwd_detached fills this buffer with the tensor-core forward kernel, one wave of tiles (at
 * most one per SM) at a time, so its size is independent of K.  Networks: 2 hidden layers of width <= 32 (31). */
int pspde_grad_from_ckpt(const pspde_cfg* cfg, const float* theta, const float* ckpt, int n_slots, int s0,
                         float* grad_theta, void* workspace, size_t workspace_bytes, void* stream);

/* Single-rollout training step for detach_forward=True (solver.py:433-499 + :221 without recomputing the trajectories,
 * like the reference, whose autograd graph keeps every activation).  pspde_rollout_fwd_ckpt is pspde_rollout_fwd_diag
 * that additionally leaves the operand rows [a0 | h1 | h2 | zeta_unit] of its first ckpt_bytes / tile_bytes tiles of
 * 128 paths in `ckpt` (layout as above, slot = tile; zeta_unit = sqrt(dt) xi_{n+1}; tile_bytes = N * C * 512);
 * pspde_grad_from_fwd_ckpt then forms
 *   dLoss/dtheta = sum_{k,n} J_theta Z' (wY_k zeta_unit)
 * with the tensor-core gradient kernel over those rows, and runs the wave-checkpointed backward of
 * pspde_rollout_bwd_detached for the tiles the buffer did not hold (prob / x0 / xi are needed only then).  With the
 * whole batch in the buffer an iteration is one forward and one gradient launch instead of forward + checkpoint
 * rollout + gradient.  Requirements (pspde_fwd_ckpt_bytes returns 0 otherwise and the caller uses
 * pspde_rollout_fwd_diag + pspde_rollout_bwd_detached): tensor-core shape class, cfg->adaptive != 0, no cotangent on
 * Z_sum (dLoss/dZsum == 0: log-variance, moment, variance, cross-entropy losses with the adaptive process).
 * pspde_fwd_ckpt_bytes = bytes for ALL ceil(K_local / 128) tiles: a K x N tape (C2: 7.1 GB, C5: 228 GB), so the caller
 * bounds it (pspde.fused: 8 GB by default) and passes what it affords, the same buffer and size to both calls.  ckpt == NULL in pspde_rollout_fwd_ckpt is the plain forward.
 * Paths with wY == 0 contribute nothing (even if they diverged).
 * With in-kernel Philox noise the s0 zeta columns of a row are NOT written (the row layout and C stay as above): zeta_unit
 * is a function of (path, step, Philox key) alone and pspde_grad_from_fwd_ckpt -- like the wave-checkpointed backward when
 * dLoss/dZsum == 0 and cfg->adaptive != 0 -- regenerates wY_k zeta_unit inside the gradient kernel (grad_tc2_kernel: hidden
 * cotangents and weight gradient on tcgen05, operand rows [a0 | h1 | h2] by TMA): 672 instead of 1 088 bytes per sample
 * at the C2 shape.  With injected noise the zeta columns are written and the older gradient kernel reads them. */
size_t pspde_fwd_ckpt_bytes(const pspde_cfg* cfg);
int pspde_rollout_fwd_ckpt(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                           const float* y0, const float* xi, float* X_N, float* Y_N, float* gX, float* Zsum,
                           double* stats, const pspde_udiag* diag, void* ckpt, size_t ckpt_bytes, void* workspace,
                           size_t workspace_bytes, void* stream);
int pspde_grad_from_fwd_ckpt(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                             const float* xi, const void* ckpt, size_t ckpt_bytes, const float* wY, float* grad_theta,
                             void* workspace, size_t workspace_bytes, void* stream);

/* Iteration glue in one launch each (the reference does these with a dozen element-wise torch kernels per iteration):
 *   pspde_lv_cotangents  loss value and per-path cotangent dLoss/dY_N of the log-variance (moment = 0, solver.py:167-168) or
 *                        moment (moment = 1, :165-166) loss from the statistics of pspde_rollout_fwd* (stats: 4 doubles, already
 *                        summed over the ranks; K_global = global batch).  A dropped trajectory (Y_N = NaN) gets zero weight.
 *                        wY: K_local floats; out3 = [loss, #dropped, K_eff] (device doubles).
 *   pspde_adam_flat      one torch.optim.Adam step (no weight decay / amsgrad) over a flat fp32 parameter buffer and its state
 *                        (solver.py:198-200 for every module at once); step = the 1-based step count AFTER this update. */
int pspde_lv_cotangents(int K_local, double K_global, int moment, const float* Y_N, const float* gX, const double* stats,
                        float* wY, double* out3, void* stream);
int pspde_adam_flat(int64_t n, float* theta, const float* grad, float* exp_avg, float* exp_avg_sq, double lr, double beta1,
                    double beta2, double eps, int64_t step, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Ensembles: M independent models of ONE configuration (same cfg -- problem, network geometry, K, N, dt, process --
 * and the same problem pack `prob` and u_L2 table), trained together with one launch per phase for all of them, so that
 * M small runs (the reference's notebooks train on K = 50 .. 256 paths: 1 .. 4 tiles, a few CTAs of the 148 SMs) fill
 * the GPU.  Members differ in Philox key, parameters, start point(s), y0 and optimizer settings.  Member m's result is
 * the result of the single-model entry point with key seeds[m] on its own slices: per-path outputs always bit for bit,
 * statistics and gradient bit for bit whenever M * ceil(K_local / 64) <= #SMs (see DESIGN.md, "Ensembles", for the
 * grid above that).  The ensemble entry points always run the FP32-FMA kernels (PSPDE_FWD_PATH / PSPDE_BWD_PATH are
 * ignored), in-kernel Philox noise only (noise_mode INJECT is refused with -5). */
typedef struct pspde_ensemble {
  int32_t n_models;                 /* M >= 1                                                                          */
  const uint64_t* seeds;            /* device, M Philox keys (cfg->seed is ignored)                                    */
  int64_t theta_stride;             /* floats between members in theta / grad_theta, >= pspde_theta_size(cfg)          */
  int64_t x0_stride;                /* floats between members' x0 (0 = one x0 -- a row or K_local rows -- for all)     */
} pspde_ensemble;

/* scratch bytes of pspde_ensemble_fwd / pspde_ensemble_bwd_detached for cfg and ens (0 on invalid input) */
size_t pspde_ensemble_workspace_bytes(const pspde_cfg* cfg, const pspde_ensemble* ens);

/* pspde_rollout_fwd_diag for every member in one rollout launch + one statistics launch: X_N [M][K_local][d] (nullable),
 * Y_N / gX / Zsum [M][K_local], stats [M][4] (nullable), diag->uL2 [M][K_local] (diag nullable; the table is shared).
 * x0: one row of d floats or (cfg->x0_per_path) K_local rows per member, member m at x0 + m * ens->x0_stride.
 * y0: nullable, else M device floats (member m starts Y at y0[m]). */
int pspde_ensemble_fwd(const pspde_cfg* cfg, const pspde_ensemble* ens, const float* theta, const float* prob,
                       const float* x0, const float* y0, float* X_N, float* Y_N, float* gX, float* Zsum, double* stats,
                       const pspde_udiag* diag, void* workspace, size_t workspace_bytes, void* stream);

/* pspde_rollout_bwd_detached (FP32-FMA recompute kernel) for every member in one launch + one reduction launch:
 * wY / wZ [M][K_local] (wZ nullable), grad_theta [M][theta_stride] (the first pspde_theta_size floats of each member
 * are overwritten, the rest of the stride is not touched).  -6 for a network the FMA backward refuses. */
int pspde_ensemble_bwd_detached(const pspde_cfg* cfg, const pspde_ensemble* ens, const float* theta, const float* prob,
                                const float* x0, const float* wY, const float* wZ, float* grad_theta, void* workspace,
                                size_t workspace_bytes, void* stream);

/* pspde_lv_cotangents for n_models members in one launch: Y_N / gX / wY [M][K_local], stats [M][4], out3 [M][3]. */
int pspde_ensemble_lv_cotangents(int32_t n_models, int K_local, double K_global, int moment, const float* Y_N,
                                 const float* gX, const double* stats, float* wY, double* out3, void* stream);

/* One member's Adam step as fp32 scalars, formed in double and rounded once (like the Python floats torch hands to its
 * kernels; pspde_adam_flat forms the same ones).  step 0 marks a member that is not updated. */
typedef struct pspde_adam_member {
  float lr_over_bc1, sqrt_bc2, one_minus_beta1, beta2, one_minus_beta2, eps;   /* bc_i = 1 - beta_i^step */
  int32_t step;
  int32_t reserved;
} pspde_adam_member;
/* host function: fills *out for (lr, beta1, beta2, eps, step); step 0 gives the "skip" entry */
int pspde_adam_member_make(double lr, double beta1, double beta2, double eps, int64_t step, pspde_adam_member* out);
/* pspde_adam_flat for n_models members in one launch: member m updates the n floats at m * stride of theta, grad,
 * exp_avg and exp_avg_sq with table[m] (device, n_models entries); members with table[m].step == 0 are left untouched. */
int pspde_ensemble_adam(int32_t n_models, int64_t n, int64_t stride, float* theta, const float* grad, float* exp_avg,
                        float* exp_avg_sq, const pspde_adam_member* table, void* stream);

/* Forward + backward for detach_forward=False (solver.py:451-469 without the detach, :221): per tile of paths the
 * states X_n are checkpointed to the workspace and the discrete adjoint runs backwards in time in the same kernel.
 *   - relative entropy, loss = mean(Zsum + g(X_N)) (solver.py:180): pass wY = wZ = wG = NULL and w = 1 / K_global;
 *     one launch gives outputs, statistics and the gradient.
 *   - any other loss: run pspde_rollout_fwd first, form the per-path cotangents wY = dL/dY_N, wZ = dL/dZsum,
 *     wG = dL/dg(X_N) (length K_local, any of them nullable = 0), then call this with them (w is ignored).
 * Outputs as in pspde_rollout_fwd (all nullable) plus grad_theta (overwritten). */
int pspde_rollout_attached(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                           const float* y0, const float* xi, float w, const float* wY, const float* wZ,
                           const float* wG, float* X_N, float* Y_N, float* gX, float* Zsum, double* stats,
                           float* grad_theta, void* workspace, size_t workspace_bytes, void* stream);

/* pspde_rollout_attached with the u_L2 diagnostic of pspde_rollout_fwd_diag evaluated in its forward sweep (the reference
 * logs it in every iteration, also for the attached relative-entropy setup, solver.py:491-494, :515).  diag nullable. */
int pspde_rollout_attached_diag(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                                const float* y0, const float* xi, float w, const float* wY, const float* wZ,
                                const float* wG, float* X_N, float* Y_N, float* gX, float* Zsum, double* stats,
                                const pspde_udiag* diag, float* grad_theta, void* workspace, size_t workspace_bytes,
                                void* stream);

/* Importance-sampling evaluation -- replaces the rollout of do_importance_sampling_me (utilities.py:287-359,
 * called from solver.py:521-528): forward-only simulation of the controlled process u = -Z on a time grid that
 * may differ from the training grid.  t_index[n] (device, length N, nullable) is the network's time index for
 * step n, n_net = ceil(n*dt / dt_net) as in Solver.Z_n (solver.py:360-362); the network sees t = n_net * dt_net
 * ('inner') or parameter set clamp(n_net) ('outer').  Per path: Y_N (the adaptive Y of pspde_rollout_fwd),
 * gX = g(X_N), Fint = sum_n f(X_{n+1}) dt; the log of the Girsanov-weighted integrand of utilities.py:329-335 is
 *   log w = -Fint - g(X_N) - ito - riemann/2 = Y_N - 2 Fint - g(X_N). */
int pspde_importance_sampling(const pspde_cfg* cfg, const float* theta, const float* prob, const float* x0,
                              const float* xi, const int32_t* t_index, float dt_net, float* X_N, float* Y_N,
                              float* gX, float* Fint, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Diffusion loss of GeneralSolver (solver.py:1001-1200, loss_method='diffusion', approx_method='Y',
 * boundary='unbounded', adaptive_forward_process=False, detach_forward=True; SURVEY.md A.5).
 *
 * cfg: net_id = PSPDE_NET_DENSENET with one output (the value function V, function_space.py:116-140),
 * time_mode = PSPDE_TIME_LAST (input [X, t], solver.py:1079), dims[0] = d + 1, problem_id = PSPDE_PROBLEM_HEAT
 * (b = a_diag x = 0, sigma = diag(b_diag) = sqrt(2) I, h = 0) or PSPDE_PROBLEM_ALLEN_CAHN (same with h = y - y^3: Y then
 * also collects -h(V(X_n, t_n)) dt on every active step, :1141, and the value row of step n gets the cotangent
 * cD act (-dh/dy dt) in the backward).  T_end = problem.T.  Per path k:
 *     Y = V(X_0, t_0);  for n < N:  act = !stopped & (t + dt <= T_end)                       (:1119, :1131)
 *         Y += (grad_x V(X, t) . (sigma xi_n sqrt(dt))) act      [= sum(Z * xi) sqrt(dt), :1100-1104, :1141-1142]
 *         X += (b(X) dt + sigma xi_n sqrt(dt)) act;  t += dt act;  stopped |= !act           (:1116-1117, :1145-1155)
 * Only the directional derivative of V enters, so the kernels carry a (value, tangent) row pair per path
 * instead of forming grad_x V by a reverse sweep as the reference does.
 * INJECT noise: element (step n, path k, component j) at xi[n*xi_stride_n + k*xi_stride_k + j*xi_stride_j]
 * (reference draw (K, d) per step, :1106: strides n: K*d, k: d, j: 1).  X0 is K_local x d, t0 has K_local entries.
 *
 * pspde_diffusion_fwd -- per path: V0 = V(X_0, t_0), VE = V(X_end, t_end), Y_end, X_end (K_local x d), t_end
 * (all nullable).  stats (nullable): 4 doubles: sum r^2 over finite r = VE - Y_end (:1163), number of active
 * (path, step) pairs (K_log, :1151-1152), sum r, number of non-finite r.
 * With N = 0 it evaluates V at (X0, t0): the terminal-condition term of :1063-1064 is this call on the first
 * K_boundary samples with t0 = T. */
size_t pspde_diffusion_workspace_bytes(const pspde_cfg* cfg, float T_end);
int pspde_diffusion_fwd(const pspde_cfg* cfg, float T_end, const float* theta, const float* prob, const float* X0,
                        const float* t0, const float* xi, float* V0, float* VE, float* Y_end, float* X_end,
                        float* t_end, double* stats, void* workspace, size_t workspace_bytes, void* stream);

/* Gradient of the diffusion loss -- replaces loss.backward() at solver.py:1187.  The trajectories are regenerated
 * (they do not depend on theta) and every step runs the reverse of the (value, tangent) pair.  Per-path
 * cotangents (length K_local, nullable = 0): c0 = dL/dV(X_0, t_0), cD = dL/d(each active directional derivative),
 * cE = dL/dV(X_end, t_end).  For loss = alpha_0 mean(r^2): w = 2 alpha_0 r / K, c0 = cD = -w, cE = w.
 * A path with all-zero cotangents is inert, even if it diverged (GeneralSolver drops a path with a non-finite r this way).
 * grad_theta (pspde_theta_size floats) is overwritten. */
int pspde_diffusion_bwd(const pspde_cfg* cfg, float T_end, const float* theta, const float* prob, const float* X0,
                        const float* t0, const float* xi, const float* c0, const float* cE, const float* cD,
                        float* grad_theta, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Elliptic sibling: diffusion loss of EllipticSolver (solver.py:628-790, loss_method='diffusion',
 * approx_method='Y', adaptive_forward_process=False, detach_forward=True; SURVEY.md row f4).
 *
 * cfg: net_id = PSPDE_NET_DENSENET with one output, time_mode = PSPDE_TIME_NONE (the value function sees X only,
 * solver.py:606), dims[0] = d; the problem pack supplies the drift a_diag x (0 in every reference problem) and
 * sigma = diag(b_diag).  Per path k:
 *     Y = V(X_0);  for n < N:  act = !stopped & inside                                           (:750-760)
 *         Y += (-h(X_n, V(X_n)) dt + grad V(X_n) . (sigma xi_n sqrt(dt))) act                    (:768-769, c = 0)
 *         X += (b(X) dt + sigma xi_n sqrt(dt)) act;   stopped |= !inside                         (:741-742, :772-779)
 *   PSPDE_DOMAIN_SPHERE  inside = |X_n| < radius, tested on the point BEFORE the step (:750-751)
 *   PSPDE_DOMAIN_BOX     inside = all_j (x_l <= proposal_j <= x_r); one_boundary: only proposal_j <= x_r (:755-758)
 *   PSPDE_DOMAIN_ANNULUS inside = radius_in < |X_n| < radius ('two_spheres', :752-753)
 * h functors (h_param[0..2]; r2 = |x|^2):
 *   PSPDE_H_ZERO                  h = 0
 *   PSPDE_H_EXP_LINEAR            ExponentialOnSphere (problems.py:985-986): -a y (4 a r2 + 2 d),                a = h_param[0]
 *   PSPDE_H_EXP_NONLINEAR         ExponentialOnBallNonlinear (:1021-1022): -2 a y (2 a r2 + d) + exp(2 a r2) - y^2
 *   PSPDE_H_EXP_NONLINEAR_SIN     ExponentialOnBallNonlinearSin (:1057-1058): ... + sin(exp(2 a r2) - y^2)
 *   PSPDE_H_HELMHOLTZ             Helmholtz (:1645-1648), d = 2: k^2 y + ((a_1 pi)^2 + (a_2 pi)^2 - k^2) sin(a_1 pi x_0) sin(a_2 pi x_1),
 *                                 (k, a_1, a_2) = h_param
 *   PSPDE_H_COMMITTOR             Committor (:1546-1580): h = 0; (a, c) = h_param[0..1] only enter the exact solution
 * The exact solution used by the V_L2 diagnostic (:733) is exp(a r2) (sin sin for Helmholtz, the harmonic profile
 * (a^2 - r^(2-d) a^d) / (a^2 - c^(2-d) a^d) for the committor).
 *
 * pspde_elliptic_fwd -- per path: V0 = V(X_0), VE = V(X_end), Y_end, X_end (K_local x d), VL2 = sum over the steps
 * a path entered un-stopped of (V(X_n) - v_true(X_n))^2 dt (all nullable).  stats as in pspde_diffusion_fwd.
 * With N = 0 it evaluates V at X0 (the Dirichlet boundary term of :669-670 is this call on the boundary samples).
 * pspde_elliptic_bwd -- cotangents as in pspde_diffusion_bwd; the value row of step n additionally receives
 * cD act (-dh/dy(X_n, V(X_n)) dt); a path with all-zero cotangents is inert, even if it diverged.  INJECT strides as in
 * pspde_diffusion_fwd. */
enum { PSPDE_DOMAIN_SPHERE = 1, PSPDE_DOMAIN_BOX = 2, PSPDE_DOMAIN_ANNULUS = 3 };
enum { PSPDE_H_ZERO = 0, PSPDE_H_EXP_LINEAR = 1, PSPDE_H_EXP_NONLINEAR = 2, PSPDE_H_EXP_NONLINEAR_SIN = 3,
       PSPDE_H_HELMHOLTZ = 4, PSPDE_H_COMMITTOR = 6 };
typedef struct pspde_elliptic {
  int32_t domain;        /* PSPDE_DOMAIN_*                                   */
  float   radius;        /* sphere: problem.boundary_distance                */
  float   x_l, x_r;      /* box: problem.X_l, problem.X_r                    */
  int32_t one_boundary;  /* box: problem.one_boundary                        */
  int32_t h_id;          /* PSPDE_H_*                                        */
  float   h_param[3];
  float   radius_in;     /* annulus: problem.boundary_distance_1 (radius = boundary_distance_2) */
} pspde_elliptic;

size_t pspde_elliptic_workspace_bytes(const pspde_cfg* cfg, const pspde_elliptic* ell);
int pspde_elliptic_fwd(const pspde_cfg* cfg, const pspde_elliptic* ell, const float* theta, const float* prob,
                       const float* X0, const float* xi, float* V0, float* VE, float* Y_end, float* X_end,
                       float* VL2, double* stats, void* workspace, size_t workspace_bytes, void* stream);
int pspde_elliptic_bwd(const pspde_cfg* cfg, const pspde_elliptic* ell, const float* theta, const float* prob,
                       const float* X0, const float* xi, const float* c0, const float* cE, const float* cD,
                       float* grad_theta, void* workspace, size_t workspace_bytes, void* stream);

/* Initial points of one iteration from Philox (key = cfg.seed, stream id = cfg.offset, global path index):
 * X_0 uniform in the ball of radius `radius` (solver.py:1045-1046), t_0 uniform in [0, T_end) (:1078). */
int pspde_diffusion_sample(const pspde_cfg* cfg, float radius, float T_end, float* X0, float* t0, void* stream);

/* Test hook: writes the increments the kernels would generate for cfg (Philox mode) in the layout
 * (N, K_local, d), i.e. strides (d, 1, K_local*d). */
int pspde_philox_dump(const pspde_cfg* cfg, float* xi_out, void* stream);

/* Self test of the tensor-core building block (csrc/tc_sm100.cuh): D[128 x N] = A[128 x K] . B[K x N] (row-major
 * device buffers) through tcgen05.mma kind::tf32 with the 3-pass hi/lo split that the tensor-core rollout uses.
 * K % 8 == 0, N % 16 == 0, N <= 256, 2K + N <= 512.  variant 0 is the production descriptor encoding. */
int pspde_tc_selftest(int K, int N, int variant, const float* A, const float* B, float* D, void* stream);

/* Self test of the TMA-fed operand path of the tensor-core gradient kernel (csrc/grad_tc_kernels.cuh): T is a device matrix
 * [R][128] fp32 (one row of 128 samples per column: the checkpoint layout); D[128 x N] = T[0..127] . T[rB..rB+N)' over the 128
 * samples, loaded 32 samples at a time by cp.async.bulk.tensor with CU_TENSOR_MAP_SWIZZLE_128B and multiplied by SS-mode
 * tcgen05.mma kind::tf32 (3 passes).  raw (nullable, R * 32 floats) receives the shared-memory image of the first box.
 * 128 <= R <= 256, R % 8 == 0, rB % 8 == 0, N % 16 == 0, rB + N <= R. */
int pspde_tma_selftest(int R, int rB, int N, const float* T, float* D, float* raw, void* stream);

/* Diagnostic: issue-to-completion cycles of chains of n tcgen05.mma kind::tf32 instructions over zeroed operands, for a fixed
 * list of (operand source, M, N) cases; out = device buffer of 4 x 32 uint64: per case {cycles to completion, cycles to issue,
 * n, mode << 32 | M << 16 | N}, terminated by a zero.  The numbers behind the gradient kernel's MMA shapes (DESIGN.md). */
int pspde_mma_probe(int n, unsigned long long* out, void* stream);

/* Deterministic fp32 FMA throughput probe (roofline denominator measured live by bench.py):
 * runs `iters` dependent-chain FMA rounds on every SM; returns the FLOP count launched, or <0. */
int64_t pspde_fma_probe(int iters, float* sink, void* stream);
/* mode 0 = scalar FFMA, 1 = packed FFMA2 (fma.rn.f32x2), 2 = FFMA2 and FFMA interleaved */
int64_t pspde_fma_probe_ex(int mode, int iters, float* sink, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PSPDE_H */
