// diffusion_kernels.cuh -- fused rollout for the diffusion loss of GeneralSolver (reference solver.py:1076-1163,
// SURVEY.md A.5): value network V(x, t) (DenseNet, scalar output, input [X, t]), unbounded domain, detached
// non-adaptive forward process.
//
//   Y_0 = V(X_0, t_0);  for n < N:  act = !stopped & (t + dt <= T)
//        Y += (grad_x V(X_n, t_n) . (B xi_n sqrt(dt))) act;   X += (b(X) dt + B xi_n sqrt(dt)) act;   t += dt act
//   loss = alpha_0 mean((V(X_end, t_end) - Y)^2)  (+ the terminal-condition term, a second call with N = 0)
//
// Only the DIRECTIONAL derivative of V along v = B xi sqrt(dt) enters (h == 0 for the heat equation), so every
// path carries two rows through the network: the value row a = [X | t | 1] and the tangent row a' = [v | 0 | 0]
// (forward-mode derivative).  A tile of P paths = 2P rows lives in shared memory for all N steps; rows
// [0, P) are value rows, rows [P, 2P) the tangent rows of the same paths, so a thread tile that owns rows r and
// r + P has both halves of a path for the activation epilogues.
//
// The trajectories do not depend on theta, and the per-path residual r_k = V(X_end) - Y_k needs the whole path, so
// the gradient is a second launch that regenerates the trajectories (Philox | injected xi) and, per step, runs
// the reverse of the (value, tangent) pair (oracle/manual.py::Net.vjp_tangent) with the per-path cotangents
//   c0 on V(X_0, t_0),  cD on every active directional derivative,  cE on V(X_end, t_end).
// A path whose three cotangents are all zero contributes nothing; the backward keeps it at the origin and stopped, so
// that a path the caller dropped for a non-finite residual (a diverged X_0) cannot put inf * 0 = NaN into the gradient.
// The network is too large for shared memory at the C4 size (371 KB of weights): the weights are re-laid once per
// call into a padded k4-blocked buffer in global memory (L2 resident) and streamed through the read-only path;
// the weight gradient of one tile-step is accumulated in registers (8x8 blocks over the 2P rows) and added to
// the CTA's private partial buffer, which a final kernel reduces in fixed order.
//
// Elliptic variant (EllipticSolver.train, solver.py:628-790, SURVEY row f4): the value network sees X only
// (TIME_NONE), the path stops when it leaves the domain instead of at t = T, and h(x, y) need not vanish:
//        act = !stopped & inside;   Y += (-h(X_n, V(X_n)) dt + grad V(X_n) . (B xi_n sqrt(dt))) act;   X += (...) act
//   sphere: inside = |X_n| < R, tested on the point BEFORE the step (:750-751);  square: X_l <= proposal <= X_r (:755-758);
//   two spheres: R_in < |X_n| < R (:752-753)
// V(X_n) is the value row of the pair the kernel carries anyway; in the reverse pass it receives the cotangent
// cD act (-dh/dy(X_n, V(X_n)) dt).  The V_L2 diagnostic of :733 is accumulated from the same value row.
#pragma once
#include "rollout_kernels.cuh"

namespace pspde {

enum { DOMAIN_TIME = 0, DOMAIN_SPHERE = 1, DOMAIN_BOX = 2, DOMAIN_ANNULUS = 3 };
enum { HFUN_ZERO = 0, HFUN_EXP_LINEAR = 1, HFUN_EXP_NONLINEAR = 2, HFUN_EXP_NONLINEAR_SIN = 3, HFUN_HELMHOLTZ = 4,
       HFUN_ALLEN_CAHN = 5, HFUN_COMMITTOR = 6 };

// h(x, y), dh/dy and the exact solution of the elliptic problems (problems.py:962-1064, :1614-1654); Allen-Cahn
// (parabolic, problems.py:1203-1204): h = y - y^3; Committor (:1546-1580): h = 0, only the exact solution is used.
//   r2 = |x|^2;  sx = sin(a_1 pi x_0) sin(a_2 pi x_1) (Helmholtz only);  hp = {alpha} or {k, a_1, a_2}
struct HFun {
  int id, d;
  float p0, p1, p2;
  __host__ __device__ float h(float r2, float sx, float y) const {
    const float a = p0;
    switch (id) {
      case HFUN_EXP_LINEAR:        return -a * y * (a * 4.0f * r2 + 2.0f * (float)d);
      case HFUN_EXP_NONLINEAR:     return -2.0f * a * y * (a * 2.0f * r2 + (float)d) + expf(2.0f * a * r2) - y * y;
      case HFUN_EXP_NONLINEAR_SIN: return -2.0f * a * y * (a * 2.0f * r2 + (float)d) + sinf(expf(2.0f * a * r2) - y * y);
      case HFUN_HELMHOLTZ: {
        const float pi = 3.14159265358979323846f, k2 = p0 * p0;
        return k2 * y + (p1 * pi) * (p1 * pi) * sx + (p2 * pi) * (p2 * pi) * sx - k2 * sx;
      }
      case HFUN_ALLEN_CAHN: return y - y * y * y;
      default: return 0.f;
    }
  }
  __host__ __device__ float h_y(float r2, float sx, float y) const {
    const float a = p0;
    switch (id) {
      case HFUN_EXP_LINEAR:        return -a * (a * 4.0f * r2 + 2.0f * (float)d);
      case HFUN_EXP_NONLINEAR:     return -2.0f * a * (a * 2.0f * r2 + (float)d) - 2.0f * y;
      case HFUN_EXP_NONLINEAR_SIN: return -2.0f * a * (a * 2.0f * r2 + (float)d) - 2.0f * y * cosf(expf(2.0f * a * r2) - y * y);
      case HFUN_HELMHOLTZ:         return p0 * p0;
      case HFUN_ALLEN_CAHN:        return 1.0f - 3.0f * y * y;
      default: return 0.f;
    }
  }
  __host__ __device__ float v_true(float r2, float sx) const {
    if (id == HFUN_HELMHOLTZ) return sx;
    if (id == HFUN_COMMITTOR) {      // problems.py:1578-1580 with a = p0, c = p1:  (a^2 - r^(2-d) a^d) / (a^2 - c^(2-d) a^d)
      const float a = p0, c = p1, ad = powf(a, (float)d);
      return (a * a - powf(sqrtf(r2), 2.0f - (float)d) * ad) / (a * a - powf(c, 2.0f - (float)d) * ad);
    }
    return expf(p0 * r2);
  }
};

struct DiffusionParams {
  NetGeom g;
  int K_local, k_offset, d, N;
  float dt, T_end;
  int noise_mode;
  unsigned long long seed;
  unsigned offset;
  long long xs_n, xs_k, xs_j;      // INJECT: xi[n * xs_n + k * xs_k + j * xs_j]
  int n_tiles;
  const float* wpack;              // k4-blocked padded weights (pspde_geom.h layout, offsets LayerGeom::w_off)
  const float* prob;               // functor pack of include/pspde.h (a_diag | b_diag | ...)
  const float *X0, *t0, *xi;
  float *V0, *VE, *Y_end, *X_end, *t_end;   // forward outputs (per path; X_end, t_end nullable)
  const float *c0, *cE, *cD;       // backward: per-path cotangents (nullable = 0)
  float* grad_partial;             // [gridDim.x][dw_partial_floats(g)]
  double* stats_partial;           // [gridDim.x][4]: sum r^2, #active steps, sum r, #non-finite r
  // elliptic variant
  int domain;                      // DOMAIN_*
  float radius, x_l, x_r;          // sphere (outer) radius / box bounds
  float radius_in;                 // annulus: inner radius
  int one_boundary;                // box: only the upper bound absorbs (solver.py:755-756)
  HFun hf;
  float* VL2;                      // forward output (per path, nullable): sum_n (V(X_n) - v_true(X_n))^2 dt over non-stopped steps
};

struct DiffSmem { int act, out, scal, prob, red, zero, total; };

PSPDE_HD inline DiffSmem diff_smem_layout(const NetGeom& g, int P) {
  DiffSmem s;
  int o = 0;
  s.act = o;  o += 2 * P * g.lda;
  s.out = o;  o += 2 * P * 4;
  s.scal = o; o += 12 * P;
  s.prob = o; o += 2 * ceil4(g.d);
  s.red = o;  o += 16;
  s.zero = o; o += 4;
  s.total = o;
  return s;
}

// weight-gradient partial: block b (8x8, 64 floats = 16 float4) of a CTA; float4 e4 of block b sits at
//   (((b >> 5) * 16 + e4) * 32 + (b & 31)) * 4   -> the 32 lanes of a warp (consecutive b) touch consecutive float4s
PSPDE_HD inline int dw_partial_floats(const NetGeom& g) { return ((g.n_blocks + 31) / 32) * 32 * 64; }
PSPDE_HD inline int dw_partial_index(int b, int e4) { return (((b >> 5) * 16 + e4) * 32 + (b & 31)) * 4; }

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float div_fast(float a, float b) {
#if defined(PSPDE_EMULATE)
  return a / b;
#else
  return __fdividef(a, b);
#endif
}

// ------------------------------------------------------------------------------------------------ forward GEMM
// pre[r][4ni..4ni+3] = sum_k act[r][k] W[k][4ni..]; thread tile = R strided rows x 4 columns; rows r and r + R/2 of
// a thread are the value / tangent rows of one path (R * PG / 2 == ROWS / 2).  W is read from global memory.
template <int ROWS, int R, typename Epi>
__device__ __forceinline__ void gemm_pairs_nn(const float* __restrict__ act, int lda, const float* __restrict__ W,
                                              int nng, int Kp, int warp, int lane, int nwarps, Epi&& epi) {
  constexpr int PG = ROWS / R;
  constexpr int NPP = PG / 8;
  static_assert(PG % 8 == 0 && R % 2 == 0, "row groups come in patches of 8, rows in (value, tangent) pairs");
  const int ncp = (nng + 3) >> 2;
  const int nwt = NPP * ncp;
  const int wstep = nng * 16;
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
      const float4 w0 = ldg4(wp), w1 = ldg4(wp + 4), w2 = ldg4(wp + 8), w3 = ldg4(wp + 12);
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
      for (int r = 0; r < R / 2; ++r) {
        float v[4], t[4];
        f2_unpack(acc[r][0], v[0], v[1]);         f2_unpack(acc[r][1], v[2], v[3]);
        f2_unpack(acc[r + R / 2][0], t[0], t[1]); f2_unpack(acc[r + R / 2][1], t[2], t[3]);
        epi(pi + r * PG, 4 * ni, v, t);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ reverse GEMM
// cotangent of hidden segment l+1 (activation columns seg_off[l+1] ...):
//   gbar[r][c] = sum_{m = l+1}^{L-1} sum_n delta_m[r][n] W_m[seg_off[l+1] + c][n]
// delta_m sits in place of segment m+1 (the output cotangent tile for m = L-1).  thread tile = R strided rows
// (value / tangent pairs) x C strided columns; epi(value row, column, gbar_value, gbar_tangent).
template <int ROWS, int R, int C, typename Epi>
__device__ __forceinline__ void gemm_pairs_nt(const NetGeom& g, int l, const float* __restrict__ sAct,
                                              const float* __restrict__ sOut, const float* __restrict__ wpack,
                                              int warp, int lane, int nwarps, Epi&& epi) {
  constexpr int PG = ROWS / R;
  constexpr int NPP = PG / 8;
  static_assert(PG % 8 == 0 && R % 2 == 0, "row groups come in patches of 8, rows in (value, tangent) pairs");
  const int c0 = g.seg_off[l + 1], ncols = g.seg_len[l + 1];
  const int CG = (ncols + C - 1) / C;
  const int ncp = (CG + 3) >> 2;
  const int nwt = NPP * ncp;
  for (int wt = warp; wt < nwt; wt += nwarps) {
    const int pp = wt % NPP, cp = wt / NPP;
    const int pi = pp * 8 + (lane & 7);
    const int ci = cp * 4 + (lane >> 3);
    f32x2 acc[R][C];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int j = 0; j < C; ++j) acc[r][j] = f2_zero();
    int col[C];
#pragma unroll
    for (int j = 0; j < C; ++j) { col[j] = ci + CG * j; if (col[j] >= ncols) col[j] = ncols - 1; }
    for (int m = l + 1; m < g.L; ++m) {
      const LayerGeom& y = g.layer[m];
      const bool last = (m == g.L - 1);
      const float* dp = (last ? sOut : sAct + g.seg_off[m + 1]) + pi * (last ? 4 : g.lda);
      const int ldl = last ? 4 : g.lda;
      const float* wr[C];
#pragma unroll
      for (int j = 0; j < C; ++j) {
        const int rr = c0 + col[j];                 // row of W_m = activation column (DenseNet: in_start == 0)
        wr[j] = wpack + y.w_off + (rr >> 2) * y.nng * 16 + (rr & 3) * 4;
      }
#pragma unroll 2
      for (int n = 0; n < y.Np; n += 4) {
        float4 dv[R], wv[C];
#pragma unroll
        for (int r = 0; r < R; ++r) dv[r] = ld4(dp + r * PG * ldl + n);
#pragma unroll
        for (int j = 0; j < C; ++j) wv[j] = ldg4(wr[j] + n * 4);
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
          for (int j = 0; j < C; ++j) {
            ffma2_v(acc[r][j], dv[r].x, dv[r].y, wv[j].x, wv[j].y);
            ffma2_v(acc[r][j], dv[r].z, dv[r].w, wv[j].z, wv[j].w);
          }
      }
    }
    if (ci < CG) {
#pragma unroll
      for (int j = 0; j < C; ++j) {
        const int c = ci + CG * j;
        if (c < ncols) {
#pragma unroll
          for (int r = 0; r < R / 2; ++r) {
            float a, b, ta, tb;
            f2_unpack(acc[r][j], a, b);
            f2_unpack(acc[r + R / 2][j], ta, tb);
            epi(pi + r * PG, c0 + c, a + b, ta + tb);
          }
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ weight gradient
// dW_l += rows(act)^T . rows(delta_l) over the 2P rows of the tile-step, one 8x8 block at a time in registers
// (block list and coordinates as in rollout_kernels.cuh), then added to this CTA's partial buffer.
template <int ROWS>
__device__ __forceinline__ void dw_accum_flush(const NetGeom& g, int l, const float* __restrict__ sAct,
                                               const float* __restrict__ sOut, const float* __restrict__ sZero,
                                               float* __restrict__ gp, int tid, int nthr) {
  const LayerGeom& y = g.layer[l];
  const int b_end = (l + 1 < g.L) ? g.layer[l + 1].blk_begin : g.n_blocks;
  for (int b = y.blk_begin + tid; b < b_end; b += nthr) {
    int kg, ng;
    bw_block_coords(y, b - y.blk_begin, kg, ng);
    const bool last = (l == g.L - 1);
    const int ldd = last ? 4 : g.lda, lda = g.lda;
    const float* a0p = sAct + y.in_start + 4 * kg;
    const float* d0p = (last ? sOut : sAct + g.seg_off[l + 1]) + 4 * ng;
    const bool ha = kg + y.kgh < y.nkg, hd = ng + y.ngh < y.nng;
    const float* a1p = ha ? a0p + 4 * y.kgh : sZero;
    const float* d1p = hd ? d0p + 4 * y.ngh : sZero;
    const int sa1 = ha ? lda : 0, sd1 = hd ? ldd : 0;
    f32x2 acc[32];
#pragma unroll
    for (int q = 0; q < 32; ++q) acc[q] = f2_zero();
#pragma unroll 2
    for (int p = 0; p < ROWS; ++p) {
      const float4 a0 = ld4(a0p), v0 = ld4(d0p), a1 = ld4(a1p), v1 = ld4(d1p);
      a0p += lda; a1p += sa1; d0p += ldd; d1p += sd1;
      const float ar[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        ffma2_s(acc[4 * i + 0], ar[i], v0.x, v0.y); ffma2_s(acc[4 * i + 1], ar[i], v0.z, v0.w);
        ffma2_s(acc[4 * i + 2], ar[i], v1.x, v1.y); ffma2_s(acc[4 * i + 3], ar[i], v1.z, v1.w);
      }
    }
#pragma unroll
    for (int e4 = 0; e4 < 16; ++e4) {
      // RED.128 into the CTA's private partial (one writer per element, program order per address: deterministic); the
      // load-add-store form exposed one L2 round trip per float4 (8 % of the kernel's stall samples at C4, and the barrier
      // wait of the other warps behind it)
      float x0, x1, x2, x3;
      f2_unpack(acc[2 * e4], x0, x1);
      f2_unpack(acc[2 * e4 + 1], x2, x3);
      red_add4(gp + dw_partial_index(b, e4), x0, x1, x2, x3);
    }
  }
}

// ------------------------------------------------------------------------------------------------ the kernel
template <int P, int T, bool BWD>
__global__ void __launch_bounds__(T, 1) diffusion_kernel(const DiffusionParams prm) {
  PSPDE_DYN_SMEM(smem4);
  float* smem = reinterpret_cast<float*>(smem4);
  constexpr int ROWS = 2 * P;
  constexpr int NW = T / 32;
  const NetGeom& g = prm.g;
  const DiffSmem sl = diff_smem_layout(g, P);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int d = prm.d, d4 = ceil4(d), N = prm.N, lda = g.lda;
  const int ngrp0 = g.seg_len[0] >> 2;       // float4 groups of segment 0 ([X | t | 1 | pad])
  const float dt = prm.dt, sq = sqrtf(prm.dt);
  float* sAct = smem + sl.act;
  float* sOut = smem + sl.out;
  float* sY = smem + sl.scal;        // [0] Y  [1] t  [2] act  [3] stopped  [4] c0  [5] cE  [6] cD  [7] #active steps
  float* sT = sY + P;
  float* sA = sY + 2 * P;
  float* sS = sY + 3 * P;
  float* sC0 = sY + 4 * P;
  float* sCE = sY + 5 * P;
  float* sCD = sY + 6 * P;
  float* sNA = sY + 7 * P;
  float* sR2 = sY + 8 * P;           // [8] |X_n|^2  [9] sin sin (Helmholtz)  [10] V_L2  [11] V(X_n) (backward)
  float* sSX = sY + 9 * P;
  float* sVL = sY + 10 * P;
  float* sVn = sY + 11 * P;
  const int domain = prm.domain;
  const HFun hf = prm.hf;
  const float* a_d = smem + sl.prob;
  const float* b_d = a_d + d4;
  double* sRed = reinterpret_cast<double*>(smem + sl.red);
  const bool philox = prm.noise_mode == NOISE_PHILOX;
  const int L = g.L;
  const LayerGeom& ylast = g.layer[L - 1];

  for (int q = tid; q < sl.total; q += T) smem[q] = 0.f;
  __syncthreads();
  for (int q = tid; q < 2 * d; q += T) { const int v = q / d, j = q - v * d; smem[sl.prob + v * d4 + j] = __ldg(prm.prob + q); }
  float* gp = BWD ? prm.grad_partial + (size_t)blockIdx.x * dw_partial_floats(g) : nullptr;
  __syncthreads();

  // backward: a path with c0 = cE = cD = 0 (the solvers zero the cotangents of a path whose residual is not finite) is
  // inert: it starts at the origin and is stopped from step 0, so every activation, h_y and epilogue value it produces
  // is finite and its zero cotangents add exact zeros to the weight gradient (from a diverged X_0, inf * 0 = NaN would)
  auto inert = [&](int k) {
    return BWD && (!prm.c0 || __ldg(prm.c0 + k) == 0.f) && (!prm.cE || __ldg(prm.cE + k) == 0.f) &&
           (!prm.cD || __ldg(prm.cD + k) == 0.f);
  };

  for (int tile = blockIdx.x; tile < prm.n_tiles; tile += gridDim.x) {
    // ---- tile init: value rows [X_0 | t_0 | 1 | 0] ([0 | t_0 | 1 | 0] for an inert path), tangent rows 0
    // (solver.py:1045-1046, :1078-1081)
    for (int q = tid; q < P * ngrp0 * 4; q += T) {
      const int p = q / (ngrp0 * 4), j = q - p * ngrp0 * 4, k = tile * P + p;
      float x = 0.f;
      if (k < prm.K_local) {
        if (j < d) x = inert(k) ? 0.f : __ldg(prm.X0 + (size_t)k * d + j);
        else if (j == g.seg_one[0]) x = 1.0f;
      }
      sAct[p * lda + j] = x;
      sAct[(P + p) * lda + j] = 0.f;
    }
    for (int p = tid; p < P; p += T) {
      const int k = tile * P + p;
      const bool in = k < prm.K_local;
      sY[p] = 0.f; sA[p] = 0.f; sNA[p] = 0.f; sVL[p] = 0.f;
      sT[p] = (in && prm.t0) ? __ldg(prm.t0 + k) : 0.f;
      sS[p] = (in && !inert(k)) ? 0.f : 1.f;
      sC0[p] = (BWD && in && prm.c0) ? __ldg(prm.c0 + k) : 0.f;
      sCE[p] = (BWD && in && prm.cE) ? __ldg(prm.cE + k) : 0.f;
      sCD[p] = (BWD && in && prm.cD) ? __ldg(prm.cD + k) : 0.f;
    }
    __syncthreads();

    // steps 0..N-1 plus the evaluation of V at the end point (n == N, zero direction)
    for (int n = 0; n <= N; ++n) {
      const bool step = n < N;
      // ---- (a) direction v = (B xi) sqrt(dt) into segment 0 of the tangent rows (solver.py:1106, :1116-1117; :726, :741-742)
      for (int q = tid; q < P * ngrp0; q += T) {
        const int p = q / ngrp0, jb = q - p * ngrp0, j0 = 4 * jb, k = tile * P + p;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        if (step && j0 < d && k < prm.K_local) {
          float e[4];
          if (philox) {
            const float4 e4 = philox_normal4((unsigned)(prm.k_offset + k), (unsigned)n, (unsigned)jb, prm.offset, prm.seed);
            e[0] = e4.x; e[1] = e4.y; e[2] = e4.z; e[3] = e4.w;
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i)
              e[i] = (j0 + i < d) ? __ldg(prm.xi + (long long)n * prm.xs_n + (long long)k * prm.xs_k + (long long)(j0 + i) * prm.xs_j) : 0.f;
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) if (j0 + i < d) v[i] = (b_d[j0 + i] * e[i]) * sq;
        }
        st4(sAct + (P + p) * lda + j0, make_float4(v[0], v[1], v[2], v[3]));
      }
      if (domain == DOMAIN_BOX) __syncthreads();       // the square test looks at the proposal X + b dt + v
      // ---- (b) who moves in this step (solver.py:1119, :1131, :1154-1155; elliptic :750-779); time column
      for (int p = tid; p < P; p += T) {
        const bool stopped = sS[p] != 0.f;
        bool sel;
        if (domain == DOMAIN_TIME) {
          const float t = sT[p];
          sel = (t + dt) <= prm.T_end;
          sAct[p * lda + g.t_col] = t;
        } else {
          const float* xr = sAct + p * lda;
          float r2 = 0.f;
          for (int j = 0; j < d; ++j) r2 += xr[j] * xr[j];
          sR2[p] = r2;
          if (hf.id == HFUN_HELMHOLTZ) {
            const float pi = 3.14159265358979323846f;
            sSX[p] = sinf(hf.p1 * pi * xr[0]) * sinf(hf.p2 * pi * xr[1]);
          }
          if (domain == DOMAIN_SPHERE) sel = sqrtf(r2) < prm.radius;
          else if (domain == DOMAIN_ANNULUS) sel = sqrtf(r2) > prm.radius_in && sqrtf(r2) < prm.radius;    // solver.py:752-753
          else {
            const float* vr = sAct + (P + p) * lda;
            sel = true;
            for (int j = 0; j < d; ++j) {
              const float xp = xr[j] + ((a_d[j] * xr[j]) * dt + vr[j]);
              sel = sel && (xp <= prm.x_r) && (prm.one_boundary || xp >= prm.x_l);
            }
          }
        }
        const bool act = step && !stopped && sel;
        sA[p] = act ? 1.f : 0.f;
        if (step && !sel) sS[p] = 1.f;
        if (act) sNA[p] += 1.f;
        sVn[p] = stopped ? 0.f : 1.f;        // "selection" at the start of the step (V_L2, solver.py:733); reused below
      }
      __syncthreads();

      // ---- (c) hidden layers, value and tangent rows together (function_space.py:133-140 and its derivative)
      for (int l = 0; l < L - 1; ++l) {
        const LayerGeom& y = g.layer[l];
        float* out = sAct + y.out_col;
        auto epi = [&](int rv, int n0, const float (&pv)[4], const float (&pd)[4]) {
          float h[4], dh[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float s = fmaxf(pv[q], 0.f);          // h = relu(p)^2, h' = 2 relu(p) p'
            h[q] = s * s;
            dh[q] = 2.0f * s * pd[q];
          }
          st4(out + rv * lda + n0, make_float4(h[0], h[1], h[2], h[3]));
          st4(out + (rv + P) * lda + n0, make_float4(dh[0], dh[1], dh[2], dh[3]));
        };
        gemm_pairs_nn<ROWS, 8>(sAct + y.in_start, lda, prm.wpack + y.w_off, y.nng, y.Kp, warp, lane, NW, epi);
        __syncthreads();
      }

      if (!BWD) {
        // ---- (d) output layer (scalar): V on the value rows, the directional derivative on the tangent rows
        for (int r = warp; r < ROWS; r += NW) {
          const float* ar = sAct + r * lda + ylast.in_start;
          const float* w = prm.wpack + ylast.w_off;
          float s = 0.f;
          for (int kk = lane; kk < ylast.Kp; kk += 32) s = fmaf(ar[kk], __ldg(w + (kk >> 2) * ylast.nng * 16 + (kk & 3) * 4), s);
          s = warp_sum(s);
          if (lane == 0) sOut[r * 4] = s;
        }
        __syncthreads();
        for (int p = tid; p < P; p += T) {
          const int k = tile * P + p;
          const float V = sOut[p * 4], dV = sOut[(P + p) * 4];
          if (n == 0) { sY[p] = V; if (k < prm.K_local && prm.V0) prm.V0[k] = V; }
          if (step) {
            if (domain == DOMAIN_TIME) {                       // solver.py:1141-1142
              if (sA[p] != 0.f) sY[p] += (hf.id != HFUN_ZERO ? -hf.h(0.f, 0.f, V) * dt : 0.f) + dV;
            }
            else {                                             // solver.py:768-769 (c = 0) and the V_L2 diagnostic (:733)
              const float r2 = sR2[p], sx = sSX[p];
              if (sA[p] != 0.f) sY[p] += -hf.h(r2, sx, V) * dt + dV;
              if (sVn[p] != 0.f) { const float e = V - hf.v_true(r2, sx); sVL[p] += (e * e) * dt; }
            }
          } else if (k < prm.K_local && prm.VE) prm.VE[k] = V;
        }
      } else {
        // ---- (e) reverse of the (value, tangent) pair; delta_l overwrites hidden segment l+1 in place
        if (hf.id != HFUN_ZERO && hf.id != HFUN_COMMITTOR && step) {        // V(X_n) for dh/dy (value rows only)
          for (int r = warp; r < P; r += NW) {
            const float* ar = sAct + r * lda + ylast.in_start;
            const float* w = prm.wpack + ylast.w_off;
            float s = 0.f;
            for (int kk = lane; kk < ylast.Kp; kk += 32) s = fmaf(ar[kk], __ldg(w + (kk >> 2) * ylast.nng * 16 + (kk & 3) * 4), s);
            s = warp_sum(s);
            if (lane == 0) sVn[r] = s;
          }
          __syncthreads();
        }
        for (int p = tid; p < P; p += T) {
          float cv = (n == 0 ? sC0[p] : 0.f) + (step ? 0.f : sCE[p]);
          const float cd = step ? sCD[p] * sA[p] : 0.f;
          if (hf.id != HFUN_ZERO && hf.id != HFUN_COMMITTOR && step) cv += cd * (-hf.h_y(sR2[p], sSX[p], sVn[p]) * dt);   // Y += -h(X_n, V(X_n)) dt
          sOut[p * 4] = cv;
          sOut[(P + p) * 4] = cd;
        }
        __syncthreads();
        // delta_{L-1} = output cotangent; every dW_m is taken as soon as delta_m is final, i.e. before the hidden
        // segments it reads as INPUT are overwritten by the cotangents of the layers below
        dw_accum_flush<ROWS>(g, L - 1, sAct, sOut, smem + sl.zero, gp, tid, T);
        __syncthreads();
        for (int l = L - 2; l >= 0; --l) {
          auto epi = [&](int rv, int col, float gv, float gt) {
            float* hv = sAct + rv * lda + col;
            float* ht = hv + P * lda;
            const float s = sqrt_fast(*hv);                    // relu(p); h'' p' = 2 [p > 0] p' = h' / relu(p)
            const float dv = gv * (2.0f * s) + (s > 0.f ? gt * div_fast(*ht, s) : 0.f);   // (approx sqrt / div: ~2 ulp, no slow paths)
            const float dd = gt * (2.0f * s);
            *hv = dv;
            *ht = dd;
          };
          gemm_pairs_nt<ROWS, 4, 4>(g, l, sAct, sOut, prm.wpack, warp, lane, NW, epi);
          __syncthreads();
          dw_accum_flush<ROWS>(g, l, sAct, sOut, smem + sl.zero, gp, tid, T);
          __syncthreads();
        }
      }

      // ---- (f) state update (solver.py:1116-1117, :1145-1148)
      if (step) {
        for (int q = tid; q < P * (d4 >> 2); q += T) {
          const int p = q / (d4 >> 2), jb = q - p * (d4 >> 2), j0 = 4 * jb;
          if (sA[p] != 0.f) {
            float* xr = sAct + p * lda + j0;
            const float* vr = sAct + (P + p) * lda + j0;
#pragma unroll
            for (int i = 0; i < 4; ++i) if (j0 + i < d) xr[i] = xr[i] + ((a_d[j0 + i] * xr[i]) * dt + vr[i]);
          }
        }
        __syncthreads();    // sA / sT are read above and rewritten below
        for (int p = tid; p < P; p += T) if (sA[p] != 0.f) sT[p] += dt;      // (stays 0 in the elliptic variant's outputs: unused)
      }
      __syncthreads();
    }

    // ---- tile epilogue
    if (!BWD) {
      double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
      if (tid < P) {
        const int k = tile * P + tid;
        if (k < prm.K_local) {
          const float Y = sY[tid];
          if (prm.Y_end) prm.Y_end[k] = Y;
          if (prm.t_end) prm.t_end[k] = sT[tid];
          if (prm.VL2) prm.VL2[k] = sVL[tid];
          const double r = (double)sOut[tid * 4] - (double)Y;    // V(X_end, t_end) - Y, solver.py:1163
          if (isfinite(r)) { s0 = r * r; s2 = r; } else s3 = 1.0;
          s1 = (double)sNA[tid];
        }
      }
      if (warp < (P + 31) / 32) {
        s0 = warp_sum_d(s0); s1 = warp_sum_d(s1); s2 = warp_sum_d(s2); s3 = warp_sum_d(s3);
        if (lane == 0) { atomicAdd(sRed + 0, s0); atomicAdd(sRed + 1, s1); atomicAdd(sRed + 2, s2); atomicAdd(sRed + 3, s3); }
      }
      if (prm.X_end) {
        for (int q = tid; q < P * d; q += T) {
          const int p = q / d, j = q - p * d, k = tile * P + p;
          if (k < prm.K_local) prm.X_end[(size_t)k * d + j] = sAct[p * lda + j];
        }
      }
    }
    __syncthreads();
  }
  if (!BWD && tid < 4 && prm.stats_partial) prm.stats_partial[blockIdx.x * 4 + tid] = sRed[tid];
}

// ------------------------------------------------------------------------------------------------ small kernels
// theta (reference layout) -> padded k4-blocked weights in global memory (what stage_weights does for shared memory)
static __global__ void pack_weights_kernel(const NetGeom g, const float* __restrict__ theta, float* __restrict__ wpack) {
  for (int l = 0; l < g.L; ++l) {
    const LayerGeom& y = g.layer[l];
    const int tot = y.Kp * y.Np;
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < tot; q += gridDim.x * blockDim.x) {
      const int blk = q >> 4, in = q & 15;
      const int r = 4 * (blk / y.nng) + (in >> 2), n = 4 * (blk % y.nng) + (in & 3);
      const int idx = theta_index(g, l, r, n);
      wpack[y.w_off + q] = idx >= 0 ? __ldg(theta + idx) : 0.f;
    }
  }
}

// per-CTA block partials -> grad_theta (fixed order, fp64); every theta entry belongs to exactly one block element
static __global__ void reduce_dw_kernel(const NetGeom g, const float* __restrict__ partial, int nparts,
                                        float* __restrict__ grad) {
  const int per = dw_partial_floats(g);
  const int tot = g.n_blocks * 64;
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < tot; q += gridDim.x * blockDim.x) {
    const int b = q >> 6, e = q & 63;
    int l = 0;
    while (l + 1 < g.L && b >= g.layer[l + 1].blk_begin) ++l;
    const LayerGeom& y = g.layer[l];
    int kg, ng;
    bw_block_coords(y, b - y.blk_begin, kg, ng);
    const int i = e >> 3, qq = (e >> 1) & 3, h = e & 1;   // acc[4 i + qq] holds columns (2 (qq & 1) + h) of half qq >> 1
    const int row = 4 * (i < 4 ? kg : kg + y.kgh) + (i & 3);
    const int col = 4 * (qq < 2 ? ng : ng + y.ngh) + 2 * (qq & 1) + h;
    if ((i >= 4 && kg + y.kgh >= y.nkg) || (qq >= 2 && ng + y.ngh >= y.nng)) continue;
    const int idx = theta_index(g, l, row, col);
    if (idx < 0) continue;
    const int off = dw_partial_index(b, e >> 2) + (e & 3);
    double s = 0.0;
    for (int c = 0; c < nparts; ++c) s += (double)partial[(size_t)c * per + off];
    grad[idx] = (float)s;
  }
}

// Initial points of one iteration (solver.py:1045-1046, :1078) from Philox: X_0 uniform in the ball of radius R
// (normalised Gaussian direction times U^(1/d)), t_0 uniform in [0, T).  Counter (k_global, 0xFFFFFFFF - jb', ...)
// keeps the streams disjoint from the per-step increments (which use n < N as the second counter word).
static __global__ void diffusion_sample_kernel(int K_local, int k_offset, int d, float radius, float T_end,
                                               unsigned long long seed, unsigned offset, float* __restrict__ X0,
                                               float* __restrict__ t0) {
  const int lane = threadIdx.x & 31;
  const int wglob = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const int ngrp = (d + 3) >> 2;
  for (int k = wglob; k < K_local; k += nwarps) {
    float ss = 0.f;
    for (int jb = lane; jb < ngrp; jb += 32) {
      const float4 z = philox_normal4((unsigned)(k_offset + k), 0xFFFFFFFFu, (unsigned)jb, offset, seed);
      const float zv[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) if (4 * jb + i < d) ss = fmaf(zv[i], zv[i], ss);
    }
    ss = warp_sum(ss);
    unsigned r[4];
    philox4x32_10((unsigned)(k_offset + k), 0xFFFFFFFEu, 0u, offset, (unsigned)(seed & 0xffffffffull), (unsigned)(seed >> 32), r);
    const float scale = radius / sqrtf(ss) * powf(u01(r[0]), 1.0f / (float)d);
    for (int jb = lane; jb < ngrp; jb += 32) {
      const float4 z = philox_normal4((unsigned)(k_offset + k), 0xFFFFFFFFu, (unsigned)jb, offset, seed);
      const float zv[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) if (4 * jb + i < d) X0[(size_t)k * d + 4 * jb + i] = zv[i] * scale;
    }
    if (lane == 0) t0[k] = u01(r[1]) * T_end;
  }
}

}  // namespace pspde
