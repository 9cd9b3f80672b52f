// rollout_kernels.cuh -- persistent fused Euler-Maruyama rollout for sm_100a (FP32 FMA path).
//
// One CTA owns a tile of P trajectories for all N steps (reference hot loop solver.py:440-494):
//   state X, the network activations, Z and the Brownian increment live in shared memory, the network weights
//   are staged into shared memory once per CTA (once per step in 'outer' mode), Y / Z_sum / g(X_N) are per-path
//   scalars in shared memory, the weight-gradient accumulators live in registers across the whole step loop.
// Per step the work is GEMM shaped over the tile and is done by three register-tiled FP32-FMA routines whose
// operands are all read as float4 from shared memory:
//   gemm_nn   pre[P x N_l]   = act[P x K_l] . W_l[K_l x N_l]                (forward, function_space.py:133-140)
//   gemm_nt   dh[P x H]     += delta_l[P x N_l] . W_l[hidden rows]^T        (cotangent of hidden activations)
//   bw_accum  dW_l[4x4 blk] += act[:, 4 cols]^T . delta_l[:, 4 cols]        (weight gradient, one VJP per (k, n))
// The backward kernel recomputes the rollout (detach_forward=True: X does not depend on theta; SURVEY.md A.3),
// so nothing of size K x N x d is ever written to HBM.
#pragma once
#include "../../include/pspde.h"
#include "philox.cuh"
#include "pspde_geom.h"
#include "simt.h"

namespace pspde {

enum { PROBLEM_OU = 0, PROBLEM_DW = 1, PROBLEM_HEAT = 2 };
enum { FLAG_DENSE_AB = 1 };
enum { NOISE_INJECT = 0, NOISE_PHILOX = 1 };

struct RolloutParams {
  NetGeom g;
  int K_local, k_offset, d, N;
  float dt;
  int problem_id, flags, adaptive, noise_mode, x0_per_path;
  unsigned long long seed;
  unsigned offset;
  long long xs_k, xs_j, xs_n;
  int n_tiles;         // ceil(K_local / P)
  int n_theta_total;   // n_params * (TIME_NONE ? N : 1)
  int n_img_total;     // w_floats * (TIME_NONE ? N : 1): floats of one CTA's weight-gradient partial (weight-IMAGE layout)
  int r_fwd[PSPDE_MAXL];  // paths per thread tile in gemm_nn, per layer (1, 2, 4 or 8)
  float w_attached;    // attached mode without per-path cotangents: wZ = wG = w_attached, wY = 0 (relative entropy)
  const float *theta, *prob, *x0, *y0, *xi, *wY, *wZ, *wG;
  float *X_N, *Y_N, *gX, *Zsum, *Fint;   // Fint (nullable): per-path sum_n f(X_{n+1}) dt
  const int* t_index;  // nullable: network time index of step n (importance sampling on a different grid)
  float dt_net;        // time-grid spacing of the network when t_index is given
  int n_sets;          // TIME_NONE: number of stacked parameter sets
  // u_L2 diagnostic (solver.py:491-494): u*(x, t_n) from per-step device tables, see include/pspde.h
  int u_mode;          // 0 off, 1 affine u* = U0[n][j] + U1[n][j] x_j, 2 lookup u* = tab[n][class(j)][cell(x_j)]
  const float* u_tab;
  int u_nx1, u_d1;
  float u_xb, u_dx;
  int u_quirk;         // mode 2: global index of the path whose cell is shifted by -2 (problems.py:279), or -1
  float d_abs_max;     // a trajectory with |D| = |Y_N - g(X_N)| >= d_abs_max counts as blown up: dropped like a non-finite one
                       // (pspde_cfg::d_abs_max; +inf when the caller leaves it off)
  float* uL2;          // per-path output
  double* stats_partial;  // [gridDim.x][4]
  float* grad_partial;    // FP32-FMA kernels: [gridDim.x][n_sets][w_floats], the k4-blocked layout of the shared weight image
                          // (pspde_geom.h) -- a thread's 8x8 block is then 16 aligned float4s; reduce_grad_image_kernel maps it
                          // to theta.  (The tensor-core gradient kernels keep their own accumulator layout here.)
  float* x_ckpt;          // attached mode: [gridDim.x][N][P][d] state checkpoints of the current tile
  // checkpointed detached backward (rollout_tc_kernels.cuh / grad_kernels.cuh): the tensor-core forward kernel writes,
  // for every (tile slot, step), the operand rows of the gradient accumulation, [a0 | h1 | h2 | zeta], COLUMN-major with
  // the 128 paths of the tile contiguous:  ckpt[((slot * N + n) * ckpt_cols + col) * 128 + path]  -- one 512-byte row per
  // column, the K-major operand form (K = sample) that the tensor-core gradient kernel loads by TMA without a transposition
  float* ckpt;
  int ckpt_cols;          // columns per (slot, step): 2 * s0 + 64, or s0 + 64 when the zeta columns are not written (ckpt_zeta == 0)
  int ckpt_s0;            // tensor-core width of the input segment (multiple of 8)
  int tile0;              // first 128-path tile of this wave (ckpt slot = tile - tile0)
  int ckpt_tiles;         // rollout: only tiles < ckpt_tiles (launch-local index) write their rows
  int ckpt_unit;          // 1: the checkpoint was written by the FORWARD pass with unit cotangents (zeta = sqrt(dt) xi);
                          //    the gradient kernel scales the zeta rows by wY[path] (adaptive, wZ == 0 only)
  int ckpt_zeta;          // 1: the zeta columns are in the checkpoint; 0: they are NOT written -- zeta = wY sqrt(dt) xi is a
                          //    function of (path, step, Philox key) alone (adaptive process, no cotangent on Z_sum, in-kernel
                          //    noise), so the gradient kernel regenerates it: 38 % less checkpoint traffic at the C2 shape
  const int* th_tbl;      // FP32-FMA kernels, nullable: (theta index, column stride | valid columns << 28) of every float4 of the
                          // shared k4-blocked weight image (theta_table_fill() below); 'outer' mode restages the weights and flushes
                          // the weight gradient EVERY step, and evaluating theta_index() there cost more than the network itself
                          // (C1: 28 k of 78 k cycles per step in the flush alone)
  const uint8_t* wpack;   // tensor-core rollout: shared-memory image of the six weight tiles in global memory (one bulk copy per
                          // CTA), or nullptr = every CTA stages its tiles from theta
  unsigned long long* prof;  // debug: per-phase clock64() totals of CTA 0 (16 slots) or nullptr
  // FP32-FMA rollout_kernel, ensemble of independent models (pspde_ensemble_*): the 1-D grid is n_models consecutive groups
  // of grid_x CTAs; CTA b serves member m = b / grid_x with the tiles b % grid_x, + grid_x, ... -- the tiles a standalone
  // launch of grid_x CTAs gives its CTAs.  Member m reads theta + m theta_stride, x0 + m x0_stride, y0[m], wY / wZ at
  // m K_local, Philox key seeds[m], and writes its per-path outputs at m K_local; its stats / gradient partials are rows
  // b of stats_partial / grad_partial, i.e. a [member][cta] slice.  grid_x = 0: one model (grid_x = gridDim.x, key seed).
  int grid_x;
  long long theta_stride, x0_stride;
  const unsigned long long* seeds;
};

// A trajectory stays in the batch if its D = Y_N - g(X_N) and Z_sum are finite and |D| is below the caller's blow-up bound.
// A dropped trajectory's Y_N is written as NaN so that the host-side mask (isfinite(Y_N - gX), pspde/losses.py) agrees with
// the statistics the kernel accumulated.
__device__ __forceinline__ bool path_kept(double D, float ZS, float d_abs_max) {
  return isfinite(D) && isfinite((double)ZS) && fabs(D) < (double)d_abs_max;
}
__device__ __forceinline__ float dropped_mark(float Y) { return isfinite(Y) ? NAN : Y; }

struct SmemLayout { int w, act, z, xi, delta, lam, scal, prob, red, zero, total; };

PSPDE_HD inline SmemLayout smem_layout(const NetGeom& g, int P, bool bwd, bool attached) {
  SmemLayout s;
  int o = 0;
  s.w = o;     o += g.w_floats;
  s.act = o;   o += P * g.lda;
  s.z = o;     o += P * g.ldz;
  s.xi = o;    o += P * g.ldz;
  s.delta = o; o += bwd ? P * g.ldd : 0;
  s.lam = o;   o += attached ? P * g.ldz : 0;
  s.scal = o;  o += 8 * P;
  s.prob = o;  o += 7 * ceil4(g.d);
  s.red = o;   o += 16;
  s.zero = o;  o += 4;
  s.total = o;
  return s;
}

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// sum over aligned groups of G lanes (G a power of two); every lane of the warp must call it
__device__ __forceinline__ float group_sum(float v, int G) {
  for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------------ packed FP32 FMA
// Blackwell's FFMA2 (PTX fma.rn.f32x2): two FP32 FMAs per lane in ONE issue slot.  The FP32 pipe rate is
// unchanged, but the slot that is freed lets the LDS / address instructions of the register-tiled GEMMs issue
// beside the math instead of in front of it.  ptxas encodes a {s, s} operand as a scalar-broadcast source
// (`R.F32`), so the outer-product form acc[i][j..j+1] += a_i * (b_j, b_j+1) needs no extra moves.
struct f32x2 {
#if defined(PSPDE_EMULATE)
  float lo, hi;
#else
  unsigned long long v;
#endif
};
__device__ __forceinline__ f32x2 f2_zero() {
#if defined(PSPDE_EMULATE)
  return f32x2{0.f, 0.f};
#else
  return f32x2{0ull};
#endif
}
// d += (s, s) * (b0, b1)
__device__ __forceinline__ void ffma2_s(f32x2& d, float s, float b0, float b1) {
#if defined(PSPDE_EMULATE)
  d.lo = fmaf(s, b0, d.lo); d.hi = fmaf(s, b1, d.hi);
#else
  asm("{\n\t.reg .b64 ss, bb;\n\tmov.b64 ss, {%1, %1};\n\tmov.b64 bb, {%2, %3};\n\tfma.rn.f32x2 %0, ss, bb, %0;\n\t}"
      : "+l"(d.v) : "f"(s), "f"(b0), "f"(b1));
#endif
}
// d += (a0, a1) * (b0, b1)
__device__ __forceinline__ void ffma2_v(f32x2& d, float a0, float a1, float b0, float b1) {
#if defined(PSPDE_EMULATE)
  d.lo = fmaf(a0, b0, d.lo); d.hi = fmaf(a1, b1, d.hi);
#else
  asm("{\n\t.reg .b64 aa, bb;\n\tmov.b64 aa, {%1, %2};\n\tmov.b64 bb, {%3, %4};\n\tfma.rn.f32x2 %0, aa, bb, %0;\n\t}"
      : "+l"(d.v) : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
#endif
}
__device__ __forceinline__ void f2_unpack(const f32x2& d, float& lo, float& hi) {
#if defined(PSPDE_EMULATE)
  lo = d.lo; hi = d.hi;
#else
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(d.v));
#endif
}

// Lane -> tile mapping shared by the GEMM routines: a warp covers a patch of 8 row groups x 4 column groups
// (lane & 7, lane >> 3).  A half-warp then touches 8 distinct activation rows (8 x 16 B = one 128 B wavefront)
// and 2 distinct weight float4s, so every LDS.128 costs the minimum of 2 shared-memory wavefronts; with the
// lanes laid along a single dimension the same loads cost 4 and the GEMMs become shared-memory bound.

// ------------------------------------------------------------------------------------------------ gemm_nn
// out[p][4ni..4ni+3] = sum_k act[p][k] * W[k][4ni..4ni+3]; thread tile = R strided rows x 4 contiguous outputs,
// W in the k4-blocked layout (pspde_geom.h).  Kp % 4 == 0.
template <int P, int R, typename Epi>
__device__ __forceinline__ void gemm_nn(const float* __restrict__ act, int lda, const float* __restrict__ W,
                                        int nng, int Kp, int warp, int lane, int nwarps, Epi&& epi) {
  constexpr int PG = P / R;            // row groups (multiple of 8)
  constexpr int NPP = PG / 8;          // row patches
  const int ncp = (nng + 3) >> 2;      // column patches
  const int nwt = NPP * ncp;
  const int wstep = nng * 16;          // floats per k4 step in W
  for (int wt = warp; wt < nwt; wt += nwarps) {
    const int pp = wt % NPP, cp = wt / NPP;
    const int pi = pp * 8 + (lane & 7);
    const int ni = cp * 4 + (lane >> 3);
    const bool valid = ni < nng;
    f32x2 acc[R][2];
#pragma unroll
    for (int r = 0; r < R; ++r) { acc[r][0] = f2_zero(); acc[r][1] = f2_zero(); }
    const float* ap = act + pi * lda;
    const float* wp = W + (valid ? ni : nng - 1) * 16;
#pragma unroll 2
    for (int k = 0; k < Kp; k += 4) {
      float4 a[R];
#pragma unroll
      for (int r = 0; r < R; ++r) a[r] = ld4(ap + r * PG * lda + k);
      const float4 w0 = ld4(wp), w1 = ld4(wp + 4), w2 = ld4(wp + 8), w3 = ld4(wp + 12);
      wp += wstep;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        ffma2_s(acc[r][0], a[r].x, w0.x, w0.y); ffma2_s(acc[r][1], a[r].x, w0.z, w0.w);
        ffma2_s(acc[r][0], a[r].y, w1.x, w1.y); ffma2_s(acc[r][1], a[r].y, w1.z, w1.w);
        ffma2_s(acc[r][0], a[r].z, w2.x, w2.y); ffma2_s(acc[r][1], a[r].z, w2.z, w2.w);
        ffma2_s(acc[r][0], a[r].w, w3.x, w3.y); ffma2_s(acc[r][1], a[r].w, w3.z, w3.w);
      }
    }
    if (valid) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        float o[4];
        f2_unpack(acc[r][0], o[0], o[1]);
        f2_unpack(acc[r][1], o[2], o[3]);
        epi(pi + r * PG, 4 * ni, o);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ gemm_nt
// out[p][c] = sum_n dl[p][n] * W[row0 + c][n], c < ncols; both operands contiguous along the reduction (W rows in
// the k4-blocked layout are float4-contiguous).  thread tile = R strided rows x C strided W-rows.  Nred % 4 == 0.
template <int P, int R, int C, typename Epi>
__device__ __forceinline__ void gemm_nt(const float* __restrict__ dl, int ldl, const float* __restrict__ W, int nng,
                                        int row0, int Nred, int ncols, int warp, int lane, int nwarps, Epi&& epi) {
  constexpr int PG = P / R;
  constexpr int NPP = PG / 8;
  const int CG = (ncols + C - 1) / C;
  const int ncp = (CG + 3) >> 2;
  const int nwt = NPP * ncp;
  for (int wt = warp; wt < nwt; wt += nwarps) {
    const int pp = wt % NPP, cp = wt / NPP;
    const int pi = pp * 8 + (lane & 7);
    const int ci = cp * 4 + (lane >> 3);
    f32x2 acc[R][C];
    const float* wr[C];
#pragma unroll
    for (int j = 0; j < C; ++j) {
      int c = ci + CG * j;
      if (c >= ncols) c = ncols - 1;
      const int rr = row0 + c;
      wr[j] = W + (rr >> 2) * nng * 16 + (rr & 3) * 4;
#pragma unroll
      for (int r = 0; r < R; ++r) acc[r][j] = f2_zero();
    }
    const float* dp = dl + pi * ldl;
#pragma unroll 2
    for (int n = 0; n < Nred; n += 4) {
      float4 dv[R], wv[C];
#pragma unroll
      for (int r = 0; r < R; ++r) dv[r] = ld4(dp + r * PG * ldl + n);
#pragma unroll
      for (int j = 0; j < C; ++j) wv[j] = ld4(wr[j] + n * 4);      // 4 columns further = next 16-float block
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < C; ++j) {
          ffma2_v(acc[r][j], dv[r].x, dv[r].y, wv[j].x, wv[j].y);
          ffma2_v(acc[r][j], dv[r].z, dv[r].w, wv[j].z, wv[j].w);
        }
    }
    if (ci < CG) {
#pragma unroll
      for (int j = 0; j < C; ++j) {
        const int c = ci + CG * j;
        if (c < ncols) {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            float lo, hi;
            f2_unpack(acc[r][j], lo, hi);
            epi(pi + r * PG, c, lo + hi);
          }
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ weight gradient
// dW_l += act^T . delta_l, accumulated in registers across the whole step loop.  Block b of the global list ->
// (layer, kg, ng) owning the 4-row groups {kg, kg + kgh} x the 4-col groups {ng, ng + ngh} (64 accumulators).
// Block -> thread assignment.  Whole warps take one block per lane over all P rows; the nb % 32 leftover blocks are
// split along the row (trajectory) dimension over the lanes of the otherwise idle warps, so that no SMSP carries
// an extra full-length warp for a handful of blocks (SMSP loads 3/3/3/3 + a sliver instead of 4/3/3/3 at C2).
// A leftover block is split into cpb = 2^k row chunks held by cpb ADJACENT lanes of one warp; the flush combines
// them with a fixed xor-shuffle butterfly, so the result stays bitwise deterministic.
// cpb > 1: this WARP holds row-split blocks (uniform per warp); a lane then owns the rows p_lo, p_lo + cpb, ... of its block.
// (Interleaved, not contiguous chunks: neighbouring lanes then read neighbouring rows of the activation and cotangent tiles,
// like the quarter-warps of gemm_nn; with contiguous chunks they sat P / cpb rows = a multiple of 32 banks apart and every
// LDS.128 replayed cpb times -- 420 cycles per row at C1.)
struct BwSlot { int b, p_lo, p_hi, cpb, l, kg, ng; };   // (l, kg, ng): layer and block coordinates of block b, found once

__device__ __forceinline__ BwSlot bw_slot_rows(const NetGeom& g, int P, int tid, int nthr) {
  BwSlot s; s.b = -1; s.p_lo = 0; s.p_hi = P; s.cpb = 1; s.l = 0; s.kg = 0; s.ng = 0;
  const int nb = g.n_blocks;
  // small networks (fewer blocks than half the threads): split EVERY block's rows over cpb lanes, so that no warp walks
  // all P rows alone while the others idle (C1: 52 blocks, 256 threads -> 4 lanes x 16 rows per block)
  if (2 * nb <= nthr) {
    int cpb = 2;
    while (cpb * 2 <= 32 && cpb * 2 <= P && cpb * 2 * nb <= nthr) cpb *= 2;
    if ((tid & ~31) < nb * cpb) s.cpb = cpb;         // (a warp without any block stays out of the flush shuffles)
    if (tid < nb * cpb) { s.b = tid / cpb; s.p_lo = tid % cpb; }
    return s;
  }
  const int full = nb & ~31, rem = nb - full, lrem = nthr - full;
  if (tid < full) { s.b = tid; return s; }
  if (rem == 0 || lrem <= 0) return s;
  int cpb = 1;
  while (cpb * 2 <= 32 && cpb * 2 <= P && cpb * 2 * rem <= lrem) cpb *= 2;
  const int l = tid - full;                      // P and cpb are powers of two
  s.cpb = cpb;
  if (l < rem * cpb) { s.b = full + l / cpb; s.p_lo = l % cpb; }
  return s;
}

__device__ __forceinline__ BwSlot bw_slot(const NetGeom& g, int P, int tid, int nthr) {
  BwSlot s = bw_slot_rows(g, P, tid, nthr);
  const int b = s.b < 0 ? 0 : s.b;      // (lanes without a block still walk through the flush shuffles of a row-split warp)
  int l = 0;
  while (l + 1 < g.L && b >= g.layer[l + 1].blk_begin) ++l;
  s.l = l;
  bw_block_coords(g.layer[l], b - g.layer[l].blk_begin, s.kg, s.ng);
  return s;
}

template <int P>
__device__ __forceinline__ void bw_accum(f32x2 (&acc)[32], const NetGeom& g, const SmemLayout& sl,
                                         const float* smem, const BwSlot& slot) {
  if (slot.b < 0) return;
  const int l = slot.l, kg = slot.kg, ng = slot.ng;
  const LayerGeom& y = g.layer[l];
  const bool last = (l == g.L - 1);
  const int ldd = last ? g.ldz : g.ldd;
  const int lda = g.lda;
  const float* a0p = smem + sl.act + y.in_start + 4 * kg + slot.p_lo * lda;
  const float* d0p = smem + (last ? sl.xi : sl.delta + (y.out_col - g.hid_off)) + 4 * ng + slot.p_lo * ldd;
  // a missing half (edge block) reads the always-zero pad with stride 0
  const bool ha = kg + y.kgh < y.nkg, hd = ng + y.ngh < y.nng;
  const float* a1p = ha ? a0p + 4 * y.kgh : smem + sl.zero;
  const float* d1p = hd ? d0p + 4 * y.ngh : smem + sl.zero;
  const int step = slot.cpb, sa0 = step * lda, sd0 = step * ldd;
  const int sa1 = ha ? sa0 : 0, sd1 = hd ? sd0 : 0;
#pragma unroll 2
  for (int p = slot.p_lo; p < slot.p_hi; p += step) {
    const float4 a0 = ld4(a0p), v0 = ld4(d0p), a1 = ld4(a1p), v1 = ld4(d1p);
    a0p += sa0; a1p += sa1; d0p += sd0; d1p += sd1;
    const float ar[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      ffma2_s(acc[4 * i + 0], ar[i], v0.x, v0.y); ffma2_s(acc[4 * i + 1], ar[i], v0.z, v0.w);
      ffma2_s(acc[4 * i + 2], ar[i], v1.x, v1.y); ffma2_s(acc[4 * i + 3], ar[i], v1.z, v1.w);
    }
  }
}

#if defined(PSPDE_EMULATE)
#define PSPDE_NOINLINE
#else
#define PSPDE_NOINLINE __noinline__
#endif

// p[0..3] += v (16-byte aligned global address), fire-and-forget: one RED.128 instead of a load-add-store round trip
__device__ __forceinline__ void red_add4(float* p, float v0, float v1, float v2, float v3) {
#if defined(PSPDE_EMULATE)
  p[0] += v0; p[1] += v1; p[2] += v2; p[3] += v3;
#else
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v0), "f"(v1), "f"(v2), "f"(v3) : "memory");
#endif
}

// One float4 (4 neighbouring columns of one row) of a weight-gradient block: combine the row-split lanes (fixed order), then
// add it into the CTA's private slice with ONE 16-byte RED (one writer per element and program order per address, so the
// sums stay bitwise deterministic).  The slice is in weight-image layout, so the float4 is aligned; in theta layout the same
// flush took 64 scalar REDs per thread, which in 'outer' mode (a flush every step into a 9 KB slice) queued up in a few L2
// slices: 16 k cycles per flush at C1.
// NOT inlined on purpose: unrolled per flush (and the flush twice per kernel) this tail was 5 k instructions, and 'outer'
// mode, which runs every phase of the kernel once per step, then spends its time in instruction fetch.
static __device__ PSPDE_NOINLINE void bw_flush_quad(float v0, float v1, float v2, float v3, int cpb, float* p, bool write) {
  for (int o = 1; o < cpb; o <<= 1) {
    v0 += __shfl_xor_sync(0xffffffffu, v0, o);
    v1 += __shfl_xor_sync(0xffffffffu, v1, o);
    v2 += __shfl_xor_sync(0xffffffffu, v2, o);
    v3 += __shfl_xor_sync(0xffffffffu, v3, o);
  }
  if (write) red_add4(p, v0, v1, v2, v3);
}

// acc -> grad_partial (this CTA's private slice, weight-image layout), then clear.  Must be called by all lanes of a warp
// (row-split warps combine their chunks with shuffles first).
__device__ __forceinline__ void bw_flush(f32x2 (&acc)[32], const NetGeom& g, const BwSlot& slot,
                                         float* __restrict__ gimg, int lane) {
  if (slot.cpb == 1 && slot.b < 0) return;      // whole warp idle or plain lane without a block
  const LayerGeom& y = g.layer[slot.l];
  const int kg = slot.kg, ng = slot.ng;
  const bool writer = slot.b >= 0 && (slot.cpb == 1 || (lane & (slot.cpb - 1)) == 0);
  const int nng = y.nng;
  const bool okn[2] = {writer, writer && ng + y.ngh < nng};
  const bool okk[2] = {true, kg + y.kgh < y.nkg};
  // image offset of (row 4 kgx + r, columns 4 ngx ..): w_off + ((kgx * nng + ngx) * 4 + r) * 4
  float* base = gimg + y.w_off;
  const int o_k[2] = {kg * nng, (kg + y.kgh) * nng}, o_n[2] = {ng, ng + y.ngh};
#pragma unroll
  for (int i = 0; i < 8; ++i) {
#pragma unroll
    for (int hq = 0; hq < 2; ++hq) {
      float v0, v1, v2, v3;
      f2_unpack(acc[4 * i + 2 * hq], v0, v1);
      f2_unpack(acc[4 * i + 2 * hq + 1], v2, v3);
      acc[4 * i + 2 * hq] = f2_zero();
      acc[4 * i + 2 * hq + 1] = f2_zero();
      bw_flush_quad(v0, v1, v2, v3, slot.cpb, base + ((o_k[i >> 2] + o_n[hq]) * 4 + (i & 3)) * 4, okk[i >> 2] && okn[hq]);
    }
  }
}

// weight-image partials of all CTAs -> theta layout: one thread per (parameter set, float4 of the image); the CTAs are summed
// in index order (deterministic).  tbl = RolloutParams::th_tbl.  Every parameter is the image of exactly one entry.
// Ensemble: n_models members, member m's nparts partials follow those of member m - 1 and its gradient goes to
// out + m out_stride.
static __global__ void reduce_grad_image_kernel(const float* __restrict__ partial, int nparts, int n_sets, int w4,
                                                const int* __restrict__ tbl, int n_params, float* __restrict__ out,
                                                int n_models, long long out_stride) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  const int per = n_sets * w4;
  if (q >= n_models * per) return;
  const int mem = q / per, r = q - mem * per;
  const int set = r / w4, q4 = r - set * w4;
  const int b0 = tbl[2 * q4], cs = tbl[2 * q4 + 1];
  if (b0 < 0) return;
  partial += (size_t)mem * nparts * per * 4;
  float s[4] = {0.f, 0.f, 0.f, 0.f};
  for (int c = 0; c < nparts; ++c) {
    const float* v = partial + (((size_t)c * n_sets + set) * w4 + q4) * 4;
    s[0] += v[0]; s[1] += v[1]; s[2] += v[2]; s[3] += v[3];
  }
  const int nv = cs >> 28, st = cs & 0x0fffffff;
  float* o = out + (size_t)mem * out_stride + (size_t)set * n_params + b0;
  for (int c = 0; c < nv; ++c) o[c * st] = s[c];
}

// (theta index, column stride | valid columns << 28) for every float4 of the shared weight image: what stage_weights and
// bw_flush otherwise derive per element with theta_index().  tbl holds 2 * (g.w_floats / 4) ints; built once per network
// geometry on the host (api_core.cu: pspde_theta_table).
inline void theta_table_fill(const NetGeom& g, int* tbl) {
  for (int l = 0; l < g.L; ++l) {
    const LayerGeom& y = g.layer[l];
    const int tot4 = (y.Kp * y.Np) >> 2;
    for (int q4 = 0; q4 < tot4; ++q4) {
      const int blk = q4 >> 2;
      const int r = 4 * (blk / y.nng) + (q4 & 3), n0 = 4 * (blk % y.nng);
      const int b0 = theta_index(g, l, r, n0);
      const int b1 = n0 + 1 < y.N ? theta_index(g, l, r, n0 + 1) : -1;
      const int cs = b1 >= 0 ? b1 - b0 : 1;
      const int nv = b0 >= 0 ? (y.N - n0 < 4 ? y.N - n0 : 4) : 0;
      int* e = tbl + 2 * ((y.w_off >> 2) + q4);
      e[0] = b0; e[1] = cs | (nv << 28);
    }
  }
}

// ------------------------------------------------------------------------------------------------ staging
// theta (one parameter set, reference layout) -> shared k4-blocked W_l with zero pads.
__device__ __forceinline__ void stage_weights(const NetGeom& g, const float* __restrict__ th, float* sW, int tid,
                                              int nthr, const int* __restrict__ tbl = nullptr) {
  if (tbl) {       // one (index, stride) pair per float4 of the image; the image is contiguous over the layers
    const int tot4 = g.w_floats >> 2;
    for (int q4 = tid; q4 < tot4; q4 += nthr) {
      const int b0 = __ldg(tbl + 2 * q4), cs = __ldg(tbl + 2 * q4 + 1);
      float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
      if (b0 >= 0) {
        const int nv = cs >> 28, st = cs & 0x0fffffff;  // valid columns of this float4 (1..4), column stride
        w.x = __ldg(th + b0);
        if (nv > 1) w.y = __ldg(th + b0 + st);
        if (nv > 2) w.z = __ldg(th + b0 + 2 * st);
        if (nv > 3) w.w = __ldg(th + b0 + 3 * st);
      }
      st4(sW + 4 * q4, w);
    }
    return;
  }
  for (int l = 0; l < g.L; ++l) {
    const LayerGeom& y = g.layer[l];
    const int tot4 = (y.Kp * y.Np) >> 2;
    for (int q4 = tid; q4 < tot4; q4 += nthr) {    // 4 q4 = shared offset of one row of a 4x4 block: 4 consecutive columns
      const int blk = q4 >> 2;
      const int r = 4 * (blk / y.nng) + (q4 & 3), n0 = 4 * (blk % y.nng);
      // theta_index is affine in the column for a fixed row: two evaluations per 4 elements ('outer' mode stages every step)
      const int b0 = theta_index(g, l, r, n0);
      const int b1 = n0 + 1 < y.N ? theta_index(g, l, r, n0 + 1) : -1;
      const int cs = b1 >= 0 ? b1 - b0 : 1;
#pragma unroll
      for (int c = 0; c < 4; ++c)
        sW[y.w_off + 4 * q4 + c] = (b0 >= 0 && n0 + c < y.N) ? __ldg(th + b0 + c * cs) : 0.f;
    }
  }
}

// INJECT mode: Brownian increment of step n for the tile -> sXi (pads stay zero).  In PHILOX mode the increments
// are generated in registers inside sde_step and never staged.
template <int P>
__device__ __forceinline__ void stage_noise(const RolloutParams& prm, int tile, int n, float* sXi, int tid,
                                            int nthr) {
  const int d = prm.d, ldz = prm.g.ldz;
  for (int q = tid; q < P * d; q += nthr) {
    const int p = q / d, j = q - p * d;
    const int k = tile * P + p;
    sXi[p * ldz + j] = (k < prm.K_local)
                           ? __ldg(prm.xi + (long long)k * prm.xs_k + (long long)j * prm.xs_j + (long long)n * prm.xs_n)
                           : 0.f;
  }
}

// ------------------------------------------------------------------------------------------------ SDE step
// Euler-Maruyama update of X, Y, Z_sum for the tile (solver.py:471-486), one warp per trajectory, one float4
// (4 state components, one Philox call) per lane.
//   X+ = X + (b(X) + B c) dt + (B xi) sqrt(dt),  c = -Z (adaptive) or 0
//   Y+ = Y + ((|Z|^2/2 + f(X+)) + Z.c) dt + (Z.xi) sqrt(dt)          [-h = |Z|^2/2 + f for every problem here]
//   Zsum += (|Z|^2/2 + f(X+)) dt
// BWD: the cotangent on Z, zeta = wY (sqrt(dt) xi + [!adaptive] Z dt) + wZ Z dt, goes to sXi and X+ is parked in sZ
// (the activation tile must keep X_n until the weight gradient has been accumulated).
template <int P, bool BWD>
__device__ __forceinline__ void sde_step(const RolloutParams& prm, const SmemLayout& sl, float* smem, int tile,
                                         int n, bool last, int warp, int lane, int nwarps, unsigned long long seed) {
  const NetGeom& g = prm.g;
  const int d = prm.d, d4 = ceil4(d), ngrp = d4 >> 2;
  const float dt = prm.dt, sq = sqrtf(prm.dt);
  const float* pa = smem + sl.prob;
  const float *a_d = pa, *b_d = pa + d4, *p_d = pa + 2 * d4, *r_d = pa + 3 * d4, *al = pa + 4 * d4,
              *kap = pa + 5 * d4, *eta = pa + 6 * d4;
  float* sY = smem + sl.scal;
  float* sZs = sY + P;
  float* sG = sY + 2 * P;
  const float* swY = sY + 3 * P;
  const float* swZ = sY + 4 * P;
  const bool adaptive = prm.adaptive != 0;
  const bool dense = (prm.flags & FLAG_DENSE_AB) != 0;
  const bool philox = prm.noise_mode == NOISE_PHILOX;
  const bool dw = prm.problem_id == PROBLEM_DW;
  const float kA = adaptive ? 0.f : 1.f;
  // G lanes per trajectory: a whole warp when the state needs it (or for the dense matvecs), else the smallest power of
  // two that covers the d/4 groups, so that a warp advances 32/G trajectories at once (d = 10: 8 per warp instead of 1 with
  // 3 live lanes).  The group sums below run over the same xor offsets as a full-warp sum whose other lanes hold zeros,
  // so the results do not depend on G.
  int G = 32;
  if (!dense) while (G > 1 && (G >> 1) >= ngrp) G >>= 1;
  const int ppw = 32 / G, gl = lane & (G - 1);
  for (int p = warp * ppw + lane / G; p < P; p += nwarps * ppw) {
    float* zr = smem + sl.z + p * g.ldz;
    float* xr = smem + sl.act + p * g.lda;          // X starts at column 0
    float* er = smem + sl.xi + p * g.ldz;
    const float wy = BWD ? swY[p] : 0.f, wz = BWD ? swZ[p] : 0.f;
    // BWD: a row with zero cotangents (padding, or a trajectory whose D was non-finite and was therefore given
    // zero weight by the host) is inert: its state stays where tile init put it (the origin) so that all its
    // activations remain finite and every product it adds to the weight gradient is exactly 0.
    const bool inert = BWD && wy == 0.f && wz == 0.f;
    const unsigned kglob = (unsigned)(prm.k_offset + tile * P + p);
    float zz = 0.f, zxi = 0.f, ff = 0.f, gg = 0.f, ul = 0.f;
    if (!dense) {
      for (int jb = gl; jb < ngrp; jb += G) {
        const int j0 = 4 * jb;
        const float4 z4 = ld4(zr + j0), x4 = ld4(xr + j0);
        float4 e4 = philox ? philox_normal4(kglob, (unsigned)n, (unsigned)jb, prm.offset, seed) : ld4(er + j0);
        const float4 A4 = ld4(a_d + j0), B4 = ld4(b_d + j0), P4 = ld4(p_d + j0);
        const float4 K4 = ld4(kap + j0);
        const float zv[4] = {z4.x, z4.y, z4.z, z4.w}, xv[4] = {x4.x, x4.y, x4.z, x4.w};
        float ev[4] = {e4.x, e4.y, e4.z, e4.w};
        const float av[4] = {A4.x, A4.y, A4.z, A4.w}, bv[4] = {B4.x, B4.y, B4.z, B4.w};
        const float pv[4] = {P4.x, P4.y, P4.z, P4.w}, kv[4] = {K4.x, K4.y, K4.z, K4.w};
        float xn[4], ze[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          // components >= d of the last group are the t / 1 / pad columns of the row: no noise, no control; all
          // their problem coefficients are zero, so x_new == x there and the group can be stored back whole
          const bool padc = j0 + i >= d;
          if (padc) ev[i] = 0.f;
          const float z = padc ? 0.f : zv[i], x = xv[i], e = ev[i];
          zz = fmaf(z, z, zz);
          zxi = fmaf(z, e, zxi);
          const float c = adaptive ? -z : 0.f;
          const float drift = dw ? -(4.0f * kv[i] * (x * (x * x - 1.0f))) : av[i] * x;
          xn[i] = x + (drift + bv[i] * c) * dt + (bv[i] * e) * sq;
          ff = fmaf(pv[i] * xn[i], xn[i], ff);
          ze[i] = wy * (sq * e + kA * dt * z) + wz * dt * z;
          if (!BWD && prm.u_mode != 0 && !padc) {           // (-Z - u*(X_{n+1}, t_n))^2, solver.py:492-493
            const int j = j0 + i;
            float us;
            if (prm.u_mode == 1) us = __ldg(prm.u_tab + (size_t)(2 * n) * d + j) + __ldg(prm.u_tab + (size_t)(2 * n + 1) * d + j) * xn[i];
            else {
              const float xc = fminf(fmaxf(xn[i], -prm.u_xb), prm.u_xb - 2.0f * prm.u_dx);
              int cell = (int)floorf((xc + prm.u_xb) / prm.u_dx);
              cell = cell < 0 ? 0 : (cell >= prm.u_nx1 ? prm.u_nx1 - 1 : cell);
              if ((int)kglob == prm.u_quirk) { cell -= 2; if (cell < 0) cell += prm.u_nx1; }    // `i[-1] -= 2`, problems.py:279
              us = __ldg(prm.u_tab + ((size_t)(2 * n) + (j < prm.u_d1 ? 0 : 1)) * prm.u_nx1 + cell);
            }
            const float du = -z - us;
            ul = fmaf(du, du, ul);
          }
        }
        if (last) {
          const float4 L4 = ld4(al + j0), R4 = ld4(r_d + j0), E4 = ld4(eta + j0);
          const float lv[4] = {L4.x, L4.y, L4.z, L4.w}, rv[4] = {R4.x, R4.y, R4.z, R4.w};
          const float tv[4] = {E4.x, E4.y, E4.z, E4.w};
#pragma unroll
          for (int i = 0; i < 4; ++i)
            gg += lv[i] * xn[i] + rv[i] * xn[i] * xn[i] + tv[i] * (xn[i] - 1.0f) * (xn[i] - 1.0f);
        }
        if (BWD) {
          st4(er + j0, inert ? make_float4(0.f, 0.f, 0.f, 0.f) : make_float4(ze[0], ze[1], ze[2], ze[3]));
          st4(zr + j0, inert ? x4 : make_float4(xn[0], xn[1], xn[2], xn[3]));
        } else {
          st4(xr + j0, make_float4(xn[0], xn[1], xn[2], xn[3]));
        }
      }
    } else {
      // dense A, B (off_diag != 0): matrices read through the read-only path; d <= 128
      const float* Am = prm.prob + 7 * d;
      const float* Bm = Am + d * d;
      if (philox) {   // the matvecs need the whole increment of the row: stage it first
        for (int jb = lane; jb < ngrp; jb += 32) {
          float4 e4 = philox_normal4(kglob, (unsigned)n, (unsigned)jb, prm.offset, seed);
          if (4 * jb + 1 >= d) e4.y = 0.f;
          if (4 * jb + 2 >= d) e4.z = 0.f;
          if (4 * jb + 3 >= d) e4.w = 0.f;
          st4(er + 4 * jb, e4);
        }
        __syncwarp();
      }
      float xn_loc[4], ze_loc[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = lane + 32 * q;
        xn_loc[q] = 0.f; ze_loc[q] = 0.f;
        if (i < d) {
          float dr = 0.f, bc = 0.f, bx = 0.f;
          for (int j = 0; j < d; ++j) {
            const float Aij = __ldg(Am + i * d + j), Bij = __ldg(Bm + i * d + j);
            dr = fmaf(Aij, xr[j], dr);
            bc = fmaf(Bij, adaptive ? -zr[j] : 0.f, bc);
            bx = fmaf(Bij, er[j], bx);
          }
          const float z = zr[i], e = er[i];
          zz = fmaf(z, z, zz);
          zxi = fmaf(z, e, zxi);
          const float xn = xr[i] + (dr + bc) * dt + bx * sq;
          xn_loc[q] = xn;
          ze_loc[q] = wy * (sq * e + kA * dt * z) + wz * dt * z;
          ff = fmaf(p_d[i] * xn, xn, ff);
          if (last) gg += al[i] * xn + r_d[i] * xn * xn + eta[i] * (xn - 1.0f) * (xn - 1.0f);
          if (!BWD && prm.u_mode == 1) {
            const float du = -z - (__ldg(prm.u_tab + (size_t)(2 * n) * d + i) + __ldg(prm.u_tab + (size_t)(2 * n + 1) * d + i) * xn);
            ul = fmaf(du, du, ul);
          }
        }
      }
      __syncwarp();
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = lane + 32 * q;
        if (i < d) {
          if (BWD) { er[i] = inert ? 0.f : ze_loc[q]; zr[i] = inert ? xr[i] : xn_loc[q]; }
          else xr[i] = xn_loc[q];
        }
      }
      // the float4 copy-back of the parked state covers whole groups: carry the t / 1 / pad columns along
      if (BWD) for (int i = d + lane; i < d4; i += 32) { zr[i] = xr[i]; er[i] = 0.f; }
    }
    zz = group_sum(zz, G); zxi = group_sum(zxi, G); ff = group_sum(ff, G);
    if (last) gg = group_sum(gg, G);
    if (!BWD && prm.u_mode != 0) { ul = group_sum(ul, G); if (gl == 0) sY[7 * P + p] += ul * dt; }
    if (gl == 0) {
      const float run = 0.5f * zz + ff;
      sY[p] += (run + (adaptive ? -zz : 0.f)) * dt + zxi * sq;
      sZs[p] += run * dt;
      sY[6 * P + p] += ff * dt;              // running cost alone (importance-sampling weights)
      if (last) sG[p] = gg;
    }
  }
}

// opt-in phase profiler (pspde_set_profile_buffer): thread 0 of CTA 0 adds the cycles since the last mark to slot `ph`
struct PhaseTimer {
  unsigned long long* buf; long long t;
  __device__ __forceinline__ void start(unsigned long long* b, int tid) {
#if defined(PSPDE_EMULATE)
    buf = nullptr; t = 0; (void)b; (void)tid;
#else
    buf = (b && tid == 0 && blockIdx.x == 0) ? b : nullptr; t = buf ? clock64() : 0;
#endif
  }
  __device__ __forceinline__ void mark(int ph) {
#if !defined(PSPDE_EMULATE)
    if (buf) { const long long n = clock64(); buf[ph] += (unsigned long long)(n - t); t = n; }
#else
    (void)ph;
#endif
  }
};

// ------------------------------------------------------------------------------------------------ network
// forward through all layers for the tile; hidden activations -> sAct, output Z -> sZ.  Ends with a barrier.
template <int P, int RMAX>
__device__ __forceinline__ void net_forward(const RolloutParams& prm, const SmemLayout& sl, float* smem, int warp,
                                            int lane, int nwarps, PhaseTimer* pt = nullptr) {
  const NetGeom& g = prm.g;
  float* sAct = smem + sl.act;
  for (int l = 0; l < g.L; ++l) {
    const LayerGeom& y = g.layer[l];
    const bool lastl = (l == g.L - 1);
    const int kind = g.kind;
    float* out = lastl ? smem + sl.z : sAct + y.out_col;
    const int ldo = lastl ? g.ldz : g.lda;
    const int N = y.N;
    auto epi = [&](int p, int n0, const float (&acc)[4]) {
      float* o = out + p * ldo + n0;
      float v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        v[q] = acc[q];
        if (!lastl) {
          if (kind == NET_DENSENET) { v[q] = fmaxf(v[q], 0.f); v[q] = v[q] * v[q]; }
          else v[q] = tanhf(v[q]);
        }
      }
      if (n0 + 3 < N) st4(o, make_float4(v[0], v[1], v[2], v[3]));
      else {
#pragma unroll
        for (int q = 0; q < 4; ++q) if (n0 + q < N) o[q] = v[q];     // never touch the 1-column / pads
      }
    };
    const float* A = sAct + y.in_start;
    const float* W = smem + sl.w + y.w_off;
    const int R = prm.r_fwd[l];
    if (RMAX >= 8 && R == 8) gemm_nn<P, (RMAX >= 8 ? 8 : 1)>(A, g.lda, W, y.nng, y.Kp, warp, lane, nwarps, epi);
    else if (RMAX >= 4 && R == 4) gemm_nn<P, (RMAX >= 4 ? 4 : 1)>(A, g.lda, W, y.nng, y.Kp, warp, lane, nwarps, epi);
    else if (R == 2) gemm_nn<P, 2>(A, g.lda, W, y.nng, y.Kp, warp, lane, nwarps, epi);
    else gemm_nn<P, 1>(A, g.lda, W, y.nng, y.Kp, warp, lane, nwarps, epi);
    if (pt) pt->mark(5 + l);         // own work of layer l (before the barrier) ...
    __syncthreads();
    if (pt) pt->mark(8 + l);         // ... and the wait for the slowest warp
  }
}

// cotangents of the hidden activations: for l = L-1 .. 1, delta tile <- delta_l . W_l[hidden rows]^T, then the
// activation derivative of segment l turns it into delta_{l-1}.  sXi holds delta_{L-1} = zeta.  Barrier after
// every layer.  (Cotangent on the network INPUT is not needed in detached mode.)
template <int P>
__device__ __forceinline__ void net_backward_hidden(const RolloutParams& prm, const SmemLayout& sl, float* smem,
                                                    int warp, int lane, int nwarps) {
  const NetGeom& g = prm.g;
  float* sDl = smem + sl.delta;
  const float* sAct = smem + sl.act;
  for (int l = g.L - 1; l >= 1; --l) {
    const LayerGeom& y = g.layer[l];
    const int c_lo = (y.in_start > g.hid_off ? y.in_start : g.hid_off);  // first hidden activation column read
    const int c_hi = y.in_start + y.Kp;
    const bool accumulate = (g.kind == NET_DENSENET) && (l < g.L - 1);
    const float* dl = (l == g.L - 1) ? smem + sl.xi : sDl + (y.out_col - g.hid_off);
    const int ldl = (l == g.L - 1) ? g.ldz : g.ldd;
    const int seg_lo = g.seg_off[l], seg_n = g.dims[l];
    const int kind = g.kind, lda = g.lda, ldd = g.ldd, hid_off = g.hid_off;
    auto epi = [&](int p, int c, float v) {
      const int col = c_lo + c;  // activation column
      float* o = sDl + p * ldd + (col - hid_off);
      if (accumulate) v += *o;
      if (col >= seg_lo) {       // segment l is now complete -> apply act'
        const int i = col - seg_lo;
        if (i < seg_n) {
          const float h = sAct[p * lda + col];
          v *= (kind == NET_DENSENET) ? 2.0f * sqrt_fast(h) : (1.0f - h * h);
        } else v = 0.f;
      }
      *o = v;
    };
    gemm_nt<P, 2, 4>(dl, ldl, smem + sl.w + y.w_off, y.nng, c_lo - y.in_start, y.Np, c_hi - c_lo, warp, lane,
                     nwarps, epi);
    __syncthreads();
  }
}

// x0, wY, wZ: the model's start points and cotangents (an ensemble member's slices of prm.x0 / prm.wY / prm.wZ)
__device__ __forceinline__ void tile_init_state(const RolloutParams& prm, float* sAct, int tile, int P, bool bwd,
                                                int tid, int nthr, const float* x0, const float* wY, const float* wZ) {
  const NetGeom& g = prm.g;
  const int d = prm.d;
  for (int q = tid; q < P * d; q += nthr) {
    const int p = q / d, j = q - p * d, k = tile * P + p;
    float x = 0.f;
    if (prm.x0_per_path) { if (k < prm.K_local) x = __ldg(x0 + (size_t)k * d + j); }
    else x = __ldg(x0 + j);
    if (bwd) {   // inert rows (zero cotangents, see sde_step) sit at the origin: finite activations whatever X_0 is
      const bool live = k < prm.K_local && ((wY && __ldg(wY + k) != 0.f) || (wZ && __ldg(wZ + k) != 0.f));
      if (!live) x = 0.f;
    }
    sAct[p * g.lda + j] = x;
  }
  for (int p = tid; p < P; p += nthr)
    for (int s = 0; s < g.L; ++s) if (g.seg_one[s] >= 0) sAct[p * g.lda + g.seg_one[s]] = 1.0f;
}

// ------------------------------------------------------------------------------------------------ the kernel
// BWD = false: forward rollout, writes per-path outputs and the loss statistics.
// BWD = true : recompute rollout + accumulate dLoss/dtheta (detached mode).  NB = weight-gradient blocks/thread.
template <int P, int T, bool BWD, int NB>
__global__ void __launch_bounds__(T, 1) rollout_kernel(const RolloutParams prm) {
  PSPDE_DYN_SMEM(smem4);
  float* smem = reinterpret_cast<float*>(smem4);
  const NetGeom& g = prm.g;
  const SmemLayout sl = smem_layout(g, P, BWD, false);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = T / 32;
  const int d = prm.d, d4 = ceil4(d), N = prm.N;
  float* sAct = smem + sl.act;
  float* sY = smem + sl.scal;
  float* sZs = sY + P;
  float* sG = sY + 2 * P;
  float* swY = sY + 3 * P;
  float* swZ = sY + 4 * P;
  double* sRed = reinterpret_cast<double*>(smem + sl.red);
  const bool outer = (g.time_mode == TIME_NONE);
  const bool inject = prm.noise_mode != NOISE_PHILOX;
  // ensemble member of this CTA and the CTA's index within the member (RolloutParams::grid_x)
  const int gx = prm.grid_x > 0 ? prm.grid_x : (int)gridDim.x;
  const int mem = blockIdx.x / gx, cta = blockIdx.x - mem * gx;
  const float* theta = prm.theta + (size_t)mem * prm.theta_stride;
  const size_t mk = (size_t)mem * prm.K_local;      // the member's first per-path slot
  const unsigned long long seed = prm.seeds ? __ldg(prm.seeds + mem) : prm.seed;

  // ---- one-time: clear every tile (pads must be zero), stage problem vectors and (inner) weights
  for (int q = sl.act + tid; q < sl.total; q += T) smem[q] = 0.f;
  __syncthreads();
  for (int q = tid; q < 7 * d; q += T) { const int v = q / d, j = q - v * d; smem[sl.prob + v * d4 + j] = __ldg(prm.prob + q); }
  if (!outer) stage_weights(g, theta, smem + sl.w, tid, T);

  static_assert(NB == 1, "one 8x8 weight-gradient block per thread");
  f32x2 acc[32];
  BwSlot slot = bw_slot(g, P, tid, T);
  if (BWD) {
#pragma unroll
    for (int q = 0; q < 32; ++q) acc[q] = f2_zero();
  }
  float* gp = BWD ? prm.grad_partial + (size_t)blockIdx.x * prm.n_img_total : nullptr;
  __syncthreads();

  for (int tile = cta; tile < prm.n_tiles; tile += gx) {
    // ---- tile init (solver.py:365-376): X = X_0, Y = y0, Z_sum = 0
    tile_init_state(prm, sAct, tile, P, BWD, tid, T, prm.x0 + (size_t)mem * prm.x0_stride, prm.wY ? prm.wY + mk : nullptr,
                    prm.wZ ? prm.wZ + mk : nullptr);
    for (int p = tid; p < P; p += T) {
      const int k = tile * P + p;
      sY[p] = prm.y0 ? __ldg(prm.y0 + mem) : 0.f;
      sZs[p] = 0.f; sG[p] = 0.f; sY[6 * P + p] = 0.f; sY[7 * P + p] = 0.f;
      const bool ok = BWD && k < prm.K_local;
      swY[p] = (ok && prm.wY) ? __ldg(prm.wY + mk + k) : 0.f;
      swZ[p] = (ok && prm.wZ) ? __ldg(prm.wZ + mk + k) : 0.f;
    }
    // (no barrier needed here: the step prologue below ends with one)

    PhaseTimer pt_;
    pt_.start(prm.prof, tid);
    for (int n = 0; n < N; ++n) {
      // time column: in BWD the float4 copy-back of X_{n+1} at the end of the previous step also covers the t column
      // when d % 4 != 0; it then writes t_{n+1} itself (same thread, no race with this loop)
      const int n_net = prm.t_index ? __ldg(prm.t_index + n) : n;          // Z_n(X, t): n = ceil(t / delta_t), :360-362
      const float t_net = prm.t_index ? (float)n_net * prm.dt_net : (float)n * prm.dt;
      if (g.t_col >= 0 && (!BWD || n == 0 || g.t_col >= d4))
        for (int p = tid; p < P; p += T) sAct[p * g.lda + g.t_col] = t_net;
      if (inject) stage_noise<P>(prm, tile, n, smem + sl.xi, tid, T);
      if (outer) {
        const int set = n_net < 0 ? 0 : (n_net >= prm.n_sets ? prm.n_sets - 1 : n_net);   // clamp like :352
        stage_weights(g, theta + (size_t)set * g.n_params, smem + sl.w, tid, T, prm.th_tbl);
      }
      __syncthreads();
      pt_.mark(0);
      net_forward<P, (BWD ? 4 : 8)>(prm, sl, smem, warp, lane, NW, &pt_);
      pt_.mark(1);
      sde_step<P, BWD>(prm, sl, smem, tile, n, n == N - 1, warp, lane, NW, seed);
      __syncthreads();
      pt_.mark(2);
      if (BWD) {
        net_backward_hidden<P>(prm, sl, smem, warp, lane, NW);
        pt_.mark(3);
        bw_accum<P>(acc, g, sl, smem, slot);
        pt_.mark(11);
        if (outer) bw_flush(acc, g, slot, gp + (size_t)n * g.w_floats, lane);
        pt_.mark(12);
        __syncthreads();
        pt_.mark(4);
        for (int q = tid; q < P * (d4 >> 2); q += T) {  // X_{n+1}: parked in sZ -> activation tile
          const int p = q / (d4 >> 2), jb = q - p * (d4 >> 2);
          st4(sAct + p * g.lda + 4 * jb, ld4(smem + sl.z + p * g.ldz + 4 * jb));
          if (g.t_col >= 0 && (g.t_col >> 2) == jb) sAct[p * g.lda + g.t_col] = (float)(n + 1) * prm.dt;
        }
        // the next step's prologue barrier (or the one below) orders this copy
      }
    }
    __syncthreads();

    // ---- tile epilogue
    if (!BWD) {
      double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
      if (tid < P) {
        const int k = tile * P + tid;
        if (k < prm.K_local) {
          const float Y = sY[tid], G = sG[tid], ZS = sZs[tid];
          const double D = (double)Y - (double)G;
          const bool keep = path_kept(D, ZS, prm.d_abs_max);
          if (prm.Y_N) prm.Y_N[mk + k] = keep ? Y : dropped_mark(Y);
          if (prm.gX) prm.gX[mk + k] = G;
          if (prm.Zsum) prm.Zsum[mk + k] = ZS;
          if (prm.Fint) prm.Fint[mk + k] = sY[6 * P + tid];
          if (prm.uL2) prm.uL2[mk + k] = sY[7 * P + tid];
          if (keep) { s0 = D; s1 = D * D; s2 = (double)ZS + (double)G; }
          else s3 = 1.0;
        }
      }
      if (warp < (P + 31) / 32) {
        s0 = warp_sum_d(s0); s1 = warp_sum_d(s1); s2 = warp_sum_d(s2); s3 = warp_sum_d(s3);
        if (lane == 0) { atomicAdd(sRed + 0, s0); atomicAdd(sRed + 1, s1); atomicAdd(sRed + 2, s2); atomicAdd(sRed + 3, s3); }
      }
      if (prm.X_N) {
        for (int q = tid; q < P * d; q += T) {
          const int p = q / d, j = q - p * d, k = tile * P + p;
          if (k < prm.K_local) prm.X_N[(mk + k) * d + j] = sAct[p * g.lda + j];
        }
      }
    } else if (!outer) {
      bw_flush(acc, g, slot, gp, lane);   // one flush per tile bounds the fp32 accumulation length to P*N terms
    }
    __syncthreads();
  }
  if (!BWD && tid < 4 && prm.stats_partial) prm.stats_partial[blockIdx.x * 4 + tid] = sRed[tid];
}

// ------------------------------------------------------------------------------------------------ attached mode
// detach_forward=False (solver.py:451-469 without the detach): the control feeds back into X, so the gradient is a
// discrete adjoint lambda_n running backwards in time (SURVEY.md A.4, generalised to any loss given by per-path
// cotangents wY = dL/dY_N, wZ = dL/dZsum, wG = dL/dg(X_N); oracle/manual.py::grad_attached):
//   lambda_N = wG grad g(X_N)
//   for n = N-1 .. 0:  lambda += (wY + wZ) dt grad f(X_{n+1})
//                      zeta = wY (-Z dt + sqrt(dt) xi_{n+1}) + wZ Z dt - dt (lambda B)
//                      dtheta += J_theta Z(t_n, X_n)' zeta;  lambda += dt J_b(X_n)' lambda + J_x Z(t_n, X_n)' zeta
// Relative entropy (loss = mean(Zsum + g), solver.py:180) has constant cotangents wZ = wG = 1/K, wY = 0 and needs
// a single launch; the other losses need the batch statistics first (forward launch, then this kernel).
// Per tile: the forward sweep checkpoints X_n (P x d floats per step) to a per-CTA scratch slice, the backward
// sweep reloads them in reverse and recomputes the network; forward and backward of a tile run in the same
// kernel, so the scratch is bounded by gridDim.x * N * P * d floats whatever K is.
template <int P, int T, int NB, int MINB = 1>
__global__ void __launch_bounds__(T, MINB) rollout_attached_kernel(const RolloutParams prm) {
  PSPDE_DYN_SMEM(smem4);
  float* smem = reinterpret_cast<float*>(smem4);
  const NetGeom& g = prm.g;
  const SmemLayout sl = smem_layout(g, P, true, true);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = T / 32;
  const int d = prm.d, d4 = ceil4(d), N = prm.N;
  const float dt = prm.dt;
  float* sAct = smem + sl.act;
  float* sLam = smem + sl.lam;
  float* sY = smem + sl.scal;
  float* sZs = sY + P;
  float* sG = sY + 2 * P;
  float* swY = sY + 3 * P;   // per-path cotangents (all 0 for padding rows and dropped trajectories)
  float* swZ = sY + 4 * P;
  float* swG = sY + 5 * P;
  double* sRed = reinterpret_cast<double*>(smem + sl.red);
  const bool outer = (g.time_mode == TIME_NONE);
  const bool dense = (prm.flags & FLAG_DENSE_AB) != 0;
  const bool inject = prm.noise_mode != NOISE_PHILOX;
  const bool per_path = prm.wY != nullptr || prm.wZ != nullptr || prm.wG != nullptr;
  const float sq = sqrtf(dt);
  const float* pa = smem + sl.prob;
  const float *a_d = pa, *b_d = pa + d4, *p_d = pa + 2 * d4, *r_d = pa + 3 * d4, *al = pa + 4 * d4,
              *kap = pa + 5 * d4, *eta = pa + 6 * d4;
  const float* Am = prm.prob + 7 * d;
  const float* Bm = Am + d * d;

  for (int q = sl.act + tid; q < sl.total; q += T) smem[q] = 0.f;
  __syncthreads();
  for (int q = tid; q < 7 * d; q += T) { const int v = q / d, j = q - v * d; smem[sl.prob + v * d4 + j] = __ldg(prm.prob + q); }
  if (!outer) stage_weights(g, prm.theta, smem + sl.w, tid, T);

  static_assert(NB == 1, "one 8x8 weight-gradient block per thread");
  f32x2 acc[32];
  const BwSlot slot = bw_slot(g, P, tid, T);
#pragma unroll
  for (int q = 0; q < 32; ++q) acc[q] = f2_zero();
  float* gp = prm.grad_partial + (size_t)blockIdx.x * prm.n_img_total;
  float* ck = prm.x_ckpt + (size_t)blockIdx.x * N * P * d;
  __syncthreads();

  for (int tile = blockIdx.x; tile < prm.n_tiles; tile += gridDim.x) {
    tile_init_state(prm, sAct, tile, P, false, tid, T, prm.x0, nullptr, nullptr);
    for (int p = tid; p < P; p += T) {
      const int k = tile * P + p;
      sY[p] = prm.y0 ? __ldg(prm.y0) : 0.f; sZs[p] = 0.f; sG[p] = 0.f; sY[6 * P + p] = 0.f; sY[7 * P + p] = 0.f;
      const bool in = k < prm.K_local;
      if (per_path) {
        swY[p] = (in && prm.wY) ? __ldg(prm.wY + k) : 0.f;
        swZ[p] = (in && prm.wZ) ? __ldg(prm.wZ + k) : 0.f;
        swG[p] = (in && prm.wG) ? __ldg(prm.wG + k) : 0.f;
      } else { swY[p] = 0.f; swZ[p] = in ? prm.w_attached : 0.f; swG[p] = swZ[p]; }
    }
    __syncthreads();
    // ---------------- forward sweep
    for (int n = 0; n < N; ++n) {
      for (int q = tid; q < P * d; q += T) {  // checkpoint X_n
        const int p = q / d, j = q - p * d;
        ck[(size_t)n * P * d + q] = sAct[p * g.lda + j];
      }
      if (g.t_col >= 0) for (int p = tid; p < P; p += T) sAct[p * g.lda + g.t_col] = (float)n * dt;
      if (inject) stage_noise<P>(prm, tile, n, smem + sl.xi, tid, T);
      if (outer) stage_weights(g, prm.theta + (size_t)n * g.n_params, smem + sl.w, tid, T, prm.th_tbl);
      __syncthreads();
      net_forward<P, 4>(prm, sl, smem, warp, lane, NW);
      sde_step<P, false>(prm, sl, smem, tile, n, n == N - 1, warp, lane, NW, prm.seed);
      __syncthreads();
    }
    // ---------------- outputs + lambda_N = w grad g(X_N)
    {
      double s2 = 0.0, s3 = 0.0;
      if (tid < P) {
        const int k = tile * P + tid;
        if (k < prm.K_local) {
          const float G = sG[tid], ZS = sZs[tid];
          if (prm.gX) prm.gX[k] = G;
          if (prm.Zsum) prm.Zsum[k] = ZS;
          const double v = (double)ZS + (double)G, D = (double)sY[tid] - (double)G;
          const bool keep = isfinite(v) && path_kept(D, ZS, prm.d_abs_max);
          if (prm.Y_N) prm.Y_N[k] = keep ? sY[tid] : dropped_mark(sY[tid]);
          if (prm.uL2) prm.uL2[k] = sY[7 * P + tid];          // u_L2 diagnostic of the forward sweep (solver.py:491-494)
          if (keep) s2 = v;
          else { s3 = 1.0; swY[tid] = 0.f; swZ[tid] = 0.f; swG[tid] = 0.f; }   // dropped from the batch and counted
        }
      }
      if (warp < (P + 31) / 32) {
        s2 = warp_sum_d(s2); s3 = warp_sum_d(s3);
        if (lane == 0) { atomicAdd(sRed + 2, s2); atomicAdd(sRed + 3, s3); }
      }
      if (prm.X_N) {
        for (int q = tid; q < P * d; q += T) {
          const int p = q / d, j = q - p * d, k = tile * P + p;
          if (k < prm.K_local) prm.X_N[(size_t)k * d + j] = sAct[p * g.lda + j];
        }
      }
    }
    __syncthreads();   // weights of non-finite trajectories were zeroed above
    for (int p = warp; p < P; p += NW) {
      const float w = swG[p];
      const bool live = swY[p] != 0.f || swZ[p] != 0.f || w != 0.f;
      const float* xr = sAct + p * g.lda;
      for (int j = lane; j < d; j += 32) {
        const float x = xr[j];
        sLam[p * g.ldz + j] = live ? w * (al[j] + 2.0f * r_d[j] * x + 2.0f * eta[j] * (x - 1.0f)) : 0.f;
      }
    }
    __syncthreads();   // X_N has been copied out by the flat loop above before any row is overwritten below
    // ---------------- backward sweep (same warp-per-row mapping for every lambda update: no barrier needed
    //                  between the end of one iteration and the start of the next)
    for (int n = N - 1; n >= 0; --n) {
      // reload X_n: the checkpoint loads of four of the warp's rows are issued together (one exposed global-memory latency
      // per batch instead of one per row: the row-by-row form was 10 % of the kernel's stall samples at the C3 shape)
      if (d <= 128) {
        const float* ckn = ck + (size_t)n * P * d;
        for (int p0 = warp; p0 < P; p0 += 4 * NW) {
          float xv[4][4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int p = p0 + u * NW;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const int j = lane + 32 * c;
              xv[u][c] = (p < P && j < d) ? ckn[p * d + j] : 0.f;
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int p = p0 + u * NW;
            if (p < P) {
              const float wf = swY[p] + swZ[p];
              const bool live = swY[p] != 0.f || swZ[p] != 0.f || swG[p] != 0.f;
              float* xr = sAct + p * g.lda;
              float* lr = sLam + p * g.ldz;
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                const int j = lane + 32 * c;
                if (j < d) {
                  if (live) {
                    lr[j] += wf * dt * 2.0f * p_d[j] * xr[j];      // grad f at X_{n+1} (f = x'Px, P diagonal)
                    xr[j] = xv[u][c];                              // X_n
                  } else { lr[j] = 0.f; xr[j] = 0.f; }             // inert row: finite state, zero adjoint
                }
              }
            }
          }
        }
      } else {
        for (int p = warp; p < P; p += NW) {
          const float wf = swY[p] + swZ[p];
          const bool live = swY[p] != 0.f || swZ[p] != 0.f || swG[p] != 0.f;
          float* xr = sAct + p * g.lda;
          float* lr = sLam + p * g.ldz;
          for (int j = lane; j < d; j += 32) {
            if (live) {
              lr[j] += wf * dt * 2.0f * p_d[j] * xr[j];
              xr[j] = ck[(size_t)n * P * d + p * d + j];
            } else { lr[j] = 0.f; xr[j] = 0.f; }
          }
        }
      }
      if (g.t_col >= 0) for (int p = tid; p < P; p += T) sAct[p * g.lda + g.t_col] = (float)n * dt;
      if (inject && per_path) stage_noise<P>(prm, tile, n, smem + sl.xi, tid, T);   // xi_{n+1} enters zeta through wY
      if (outer) stage_weights(g, prm.theta + (size_t)n * g.n_params, smem + sl.w, tid, T, prm.th_tbl);
      __syncthreads();
      net_forward<P, 4>(prm, sl, smem, warp, lane, NW);
      // zeta -> sXi: no cross-lane sums here, so the (row, 4-column group) pairs are simply dealt out to all threads (a warp
      // per row left 19 of 32 lanes idle at d = 50 and walked its 8 rows one after the other)
      const int ngrp_z = (d + 3) >> 2;
      for (int q = tid; q < P * ngrp_z; q += T) {
        const int p = q / ngrp_z, jb = q - p * ngrp_z;
        const float wy = swY[p], wz = swZ[p];
        const float* zr = smem + sl.z + p * g.ldz;
        const float* lr = sLam + p * g.ldz;
        float* er = smem + sl.xi + p * g.ldz;
        const unsigned kglob = (unsigned)(prm.k_offset + tile * P + p);
        {
          float e4[4] = {0.f, 0.f, 0.f, 0.f};
          if (wy != 0.f) {
            if (inject) { const float4 t4 = ld4(er + 4 * jb); e4[0] = t4.x; e4[1] = t4.y; e4[2] = t4.z; e4[3] = t4.w; }
            else { const float4 t4 = philox_normal4(kglob, (unsigned)n, (unsigned)jb, prm.offset, prm.seed);
                   e4[0] = t4.x; e4[1] = t4.y; e4[2] = t4.z; e4[3] = t4.w; }
          }
          float o4[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int j = 4 * jb + i;
            o4[i] = 0.f;
            if (j < d) {
              float lb;
              if (!dense) lb = lr[j] * b_d[j];
              else { lb = 0.f; for (int q = 0; q < d; ++q) lb = fmaf(lr[q], __ldg(Bm + q * d + j), lb); }
              const float z = zr[j];
              o4[i] = wy * (sq * e4[i] - dt * z) + wz * dt * z - dt * lb;
            }
          }
          st4(er + 4 * jb, make_float4(o4[0], o4[1], o4[2], o4[3]));
        }
      }
      __syncthreads();
      net_backward_hidden<P>(prm, sl, smem, warp, lane, NW);
      // cotangent on X through the network input: dx = sum_l delta_l . W_l[x rows]'  -> sZ
      {
        float* sDx = smem + sl.z;
        const int ldz = g.ldz;
        const int l_hi = (g.kind == NET_DENSENET) ? g.L - 1 : 0;
        for (int l = 0; l <= l_hi; ++l) {
          const LayerGeom& y = g.layer[l];
          const float* dl = (l == g.L - 1) ? smem + sl.xi : smem + sl.delta + (y.out_col - g.hid_off);
          const int ldl = (l == g.L - 1) ? g.ldz : g.ldd;
          const bool first = (l == 0);
          auto epi = [&](int p, int c, float v) {
            float* o = sDx + p * ldz + c;
            *o = first ? v : *o + v;
          };
          gemm_nt<P, 2, 4>(dl, ldl, smem + sl.w + y.w_off, y.nng, 0, y.Np, d, warp, lane, NW, epi);   // X rows = 0..d-1
        }
      }
      bw_accum<P>(acc, g, sl, smem, slot);
      if (outer) bw_flush(acc, g, slot, gp + (size_t)n * g.w_floats, lane);
      __syncthreads();
      for (int p = warp; p < P; p += NW) {                          // lambda_n
        const float* xr = sAct + p * g.lda;
        const float* dx = smem + sl.z + p * g.ldz;
        float* lr = sLam + p * g.ldz;
        if (!dense) {
          for (int j = lane; j < d; j += 32) {
            const float x = xr[j];
            const float jb = (prm.problem_id == PROBLEM_DW) ? -4.0f * kap[j] * (3.0f * x * x - 1.0f) : a_d[j];
            lr[j] = lr[j] + dt * jb * lr[j] + dx[j];
          }
        } else {
          float ln[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int j = lane + 32 * q;
            ln[q] = 0.f;
            if (j < d) {
              float la = 0.f;
              for (int i = 0; i < d; ++i) la = fmaf(lr[i], __ldg(Am + i * d + j), la);
              ln[q] = lr[j] + dt * la + dx[j];
            }
          }
          __syncwarp();
#pragma unroll
          for (int q = 0; q < 4; ++q) { const int j = lane + 32 * q; if (j < d) lr[j] = ln[q]; }
        }
      }
    }
    if (!outer) bw_flush(acc, g, slot, gp, lane);
    __syncthreads();
  }
  if (tid < 4 && prm.stats_partial) prm.stats_partial[blockIdx.x * 4 + tid] = sRed[tid];
}

// ------------------------------------------------------------------------------------------------ small kernels
// deterministic cross-CTA reductions (fixed order, fp64 accumulation): one thread per (model, statistic), the nparts
// CTAs of a model summed in index order; model m's partials follow model m - 1's, its 4 sums go to out[4 m ..]
static __global__ void reduce_stats_kernel(const double* __restrict__ partial, int nparts, int n_models,
                                           double* __restrict__ out) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q < 4 * n_models) {
    const int mem = q >> 2, i = q & 3;
    const double* pm = partial + (size_t)mem * nparts * 4;
    double s = 0.0;
    for (int c = 0; c < nparts; ++c) s += pm[c * 4 + i];
    out[q] = s;
  }
}

// Loss value and per-path cotangents of the log-variance / moment losses (solver.py:165-168) from the batch statistics the
// forward kernel accumulated (summed over the ranks by the caller): the dozen element-wise launches of the host formulation
// in one.  stats = [sum D, sum D^2, -, #dropped] over the kept trajectories, D = Y_N - g(X_N); a dropped trajectory carries
// Y_N = NaN (path_kept) and gets zero weight.  out = [loss, #dropped, K_eff].
// Ensemble: the grid is one group of ceil(K_local / blockDim.x) blocks per model; model m has Y / gX / wY at m K_local,
// stats at 4 m and out at 3 m.
static __global__ void lv_cotangents_kernel(int K_local, double K_global, int moment, const float* __restrict__ Y,
                                            const float* __restrict__ gX, const double* __restrict__ stats,
                                            float* __restrict__ wY, double* __restrict__ out) {
  const int nb = (K_local + blockDim.x - 1) / blockDim.x, mem = blockIdx.x / nb;
  const size_t mk = (size_t)mem * K_local;
  Y += mk; gX += mk; wY += mk; stats += 4 * mem; out += 3 * mem;
  const double Ke = K_global - stats[3];
  const double mean = stats[0] / Ke;
  const int k = (blockIdx.x - mem * nb) * blockDim.x + threadIdx.x;
  if (k < K_local) {
    const double D = (double)(Y[k] - gX[k]);                   // fp32 subtraction, then widened: the host formulation's order
    wY[k] = isfinite(D) ? (float)((moment ? D : D - mean) * (2.0 / Ke)) : 0.f;
  }
  if (k == 0) { out[0] = moment ? stats[1] / Ke : stats[1] / Ke - mean * mean; out[1] = stats[3]; out[2] = Ke; }
}

// single-rounding fp32 operations (no FMA contraction): the update must follow torch's op sequence
#if defined(PSPDE_EMULATE)
static inline float rn_add(float a, float b) { volatile float r = a + b; return r; }
static inline float rn_sub(float a, float b) { volatile float r = a - b; return r; }
static inline float rn_mul(float a, float b) { volatile float r = a * b; return r; }
static inline float rn_div(float a, float b) { volatile float r = a / b; return r; }
static inline float rn_sqrt(float a) { return sqrtf(a); }
#else
__device__ __forceinline__ float rn_add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float rn_sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float rn_mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float rn_div(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ float rn_sqrt(float a) { return __fsqrt_rn(a); }
#endif
// One Adam step over a flat parameter buffer: the op sequence of torch.optim.Adam's single-tensor form (no weight decay,
// no amsgrad): m = lerp(m, g, 1 - b1); v = v b2 + (1 - b2) g g; theta -= (lr / bc1) m / (sqrt(v) / sqrt(bc2) + eps).
// Ensemble: the grid is one group of ceil(n / blockDim.x) blocks per model; model m updates the n floats at m stride of the
// four buffers with the scalars tbl[m] (tbl == nullptr: one model with `one`); a model whose step is 0 is left untouched.
static __global__ void adam_flat_kernel(int n, long long stride, float* __restrict__ theta, const float* __restrict__ g,
                                        float* __restrict__ m, float* __restrict__ v, const pspde_adam_member* __restrict__ tbl,
                                        pspde_adam_member one) {
  const int nb = (n + blockDim.x - 1) / blockDim.x, mem = blockIdx.x / nb;
  const pspde_adam_member s = tbl ? tbl[mem] : one;
  const int i = (blockIdx.x - mem * nb) * blockDim.x + threadIdx.x;
  if (s.step != 0 && i < n) {
    const size_t o = (size_t)mem * stride;
    theta += o; g += o; m += o; v += o;
    const float lr_over_bc1 = s.lr_over_bc1, sqrt_bc2 = s.sqrt_bc2, omb1 = s.one_minus_beta1, b2 = s.beta2,
                omb2 = s.one_minus_beta2, eps = s.eps;
    const float gi = g[i];
    const float mi = rn_add(m[i], rn_mul(rn_sub(gi, m[i]), omb1));
    const float vi = rn_add(rn_mul(v[i], b2), rn_mul(rn_mul(gi, gi), omb2));
    m[i] = mi; v[i] = vi;
    const float denom = rn_add(rn_div(rn_sqrt(vi), sqrt_bc2), eps);
    theta[i] = rn_sub(theta[i], rn_mul(lr_over_bc1, rn_div(mi, denom)));
  }
}

// increments the rollout kernels would draw, layout (N, K_local, d)
static __global__ void philox_dump_kernel(int K_local, int k_offset, int d, int N, unsigned long long seed, unsigned offset,
                                   float* __restrict__ out) {
  const int nb4 = (d + 3) >> 2;
  const long long total = (long long)N * K_local * nb4;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (long long)gridDim.x * blockDim.x) {
    const int jb = (int)(q % nb4);
    const long long r = q / nb4;
    const int k = (int)(r % K_local), n = (int)(r / K_local);
    const float4 z = philox_normal4((unsigned)(k_offset + k), (unsigned)n, (unsigned)jb, offset, seed);
    float* o = out + ((size_t)n * K_local + k) * d + 4 * jb;
    o[0] = z.x;
    if (4 * jb + 1 < d) o[1] = z.y;
    if (4 * jb + 2 < d) o[2] = z.z;
    if (4 * jb + 3 < d) o[3] = z.w;
  }
}

// FP32 FMA throughput probe: 8 independent chains per thread.
//   mode 0: scalar FFMA (2 FLOP each)   mode 1: packed FFMA2 (4 FLOP each)   mode 2: one FFMA2 + two FFMA interleaved
template <int MODE>
static __global__ void __launch_bounds__(1024, 1) fma_probe_kernel(int iters, float* __restrict__ sink) {
  const float m = 0.9999f, c = 1e-7f;
  float a[8];
  f32x2 b[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { a[i] = threadIdx.x * 1e-9f + i; b[i] = f2_zero(); }
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 16; ++u) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (MODE == 0) a[i] = fmaf(a[i], m, c);
        else if (MODE == 1) ffma2_s(b[i], m, a[i], c);
        else { if (i & 1) ffma2_s(b[i], m, a[i], c); else { a[i] = fmaf(a[i], m, c); a[i] = fmaf(a[i], m, c); } }
      }
    }
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) { float lo, hi; f2_unpack(b[i], lo, hi); s += a[i] + lo + hi; }
  if (s == 123.456f) sink[0] = s;
}

}  // namespace pspde
