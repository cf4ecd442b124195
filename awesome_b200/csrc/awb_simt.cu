// CUDA-core fp32 kernels of the prior-fit path (AWB_PREC_FP32): the exact-arithmetic
// implementation, comparable with the reference to fp32 rounding.  Layer contractions are
// tiled SGEMMs over the augmented activation rows (see awb_internal.cuh); every
// elementwise step of the reference (bias, skip connection, relu, relu-backward, sigmoid,
// loss, clamp) is fused into a producing kernel's epilogue.  Cross-pixel reductions
// (weight gradients, loss) are per-pixel-range partial sums reduced in a fixed order by
// the optimizer kernel: deterministic, no atomics.
#include <cuda_fp16.h>
#include <math.h>

#include "awb_internal.cuh"

namespace awb {

// ------------------------------------------------------------------ pack
// arena (state_dict order) -> augmented fp32 weights.  waug is zeroed by the caller.
__global__ void k_pack(const float* __restrict__ params, float* __restrict__ waug,
                       const int32_t* __restrict__ map, int P_icnn, int64_t P, int64_t off_icnn,
                       int64_t G) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int o = blockIdx.y;
  if (i < P_icnn) waug[o * G + map[i]] = params[o * P + off_icnn + i];
}

// ------------------------------------------------------------------ input layer (a1 + a7 first line)
// z0 = relu(W_in x + b_in)  (convex_net.py:209), written as augmented rows ZA0.
// x comes from the grid (generated in-kernel: no HBM read) or from X when a flow produced it.
__global__ void __launch_bounds__(256) k_input(GridDev g, int x_ready, float* __restrict__ X,
                                               const float* __restrict__ waug, float* __restrict__ ZA0,
                                               int64_t N, int h, int C, int ld, int64_t G, int64_t aug_in,
                                               int64_t strideZA) {
  __shared__ float xs[64][4];
  int o = blockIdx.y;
  int64_t n0 = (int64_t)blockIdx.x * 64;
  float* Xo = X + (int64_t)o * N * 4;
  if (threadIdx.x < 64) {
    int64_t n = n0 + threadIdx.x;
    float4 v = make_float4(0.f, 0.f, 0.f, 1.f);
    if (n < N) {
      if (x_ready) {
        v = *reinterpret_cast<const float4*>(Xo + n * 4);
      } else {
        v.x = coord(g, n, 0);
        v.y = coord(g, n, 1);
        v.z = C > 2 ? coord(g, n, 2) : 0.f;
        v.w = 1.f;
        *reinterpret_cast<float4*>(Xo + n * 4) = v;
      }
    }
    xs[threadIdx.x][0] = v.x; xs[threadIdx.x][1] = v.y; xs[threadIdx.x][2] = v.z; xs[threadIdx.x][3] = 1.f;
  }
  __syncthreads();
  const float* win = waug + (int64_t)o * G + aug_in;
  float* Z = ZA0 + (int64_t)o * strideZA;
  for (int idx = threadIdx.x; idx < 64 * ld; idx += 256) {
    int r = idx / ld, c = idx - r * ld;
    int64_t n = n0 + r;
    if (n >= N) break;
    float v;
    if (c < h) {
      float4 w = *reinterpret_cast<const float4*>(win + c * 4);
      // same association as addmm: bias + sum_k x_k w_k (k ascending)
      float a = xs[r][0] * w.x;
      a = fmaf(xs[r][1], w.y, a);
      if (C > 2) a = fmaf(xs[r][2], w.z, a);
      a += w.w;
      v = fmaxf(a, 0.f);
    } else if (c < h + C) {
      v = xs[r][c - h];
    } else {
      v = (c == h + C) ? 1.f : 0.f;
    }
    Z[n * ld + c] = v;
  }
}

// ------------------------------------------------------------------ tangent input layer (second-order pass)
// Tangent of the forward along u_n = d R / d dgrid_n (planar [B,C,H,W], read through gu):
// ZT0[n] = [ (W_in u) .* (z0 > 0) | u | 0 | 0-pad ] -- the bias column is the tangent of a constant -- and the rows
// (u, 0) that the input layer's weight gradient reads.  Single object.
__global__ void __launch_bounds__(256) k_tan_input(GridDev gu, const float* __restrict__ waug,
                                                   const float* __restrict__ ZA0, float* __restrict__ ZT0,
                                                   float* __restrict__ U, int64_t N, int h, int C, int ld,
                                                   int64_t aug_in) {
  __shared__ float us[64][4];
  int64_t n0 = (int64_t)blockIdx.x * 64;
  if (threadIdx.x < 64) {
    int64_t n = n0 + threadIdx.x;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (n < N) {
      v.x = gu.grid[planar_index(gu, n, 0)];
      v.y = gu.grid[planar_index(gu, n, 1)];
      v.z = C > 2 ? gu.grid[planar_index(gu, n, 2)] : 0.f;
      *reinterpret_cast<float4*>(U + n * 4) = v;
    }
    us[threadIdx.x][0] = v.x; us[threadIdx.x][1] = v.y; us[threadIdx.x][2] = v.z; us[threadIdx.x][3] = 0.f;
  }
  __syncthreads();
  const float* win = waug + aug_in;
  for (int idx = threadIdx.x; idx < 64 * ld; idx += 256) {
    int r = idx / ld, c = idx - r * ld;
    int64_t n = n0 + r;
    if (n >= N) break;
    float v;
    if (c < h) {
      float4 w = *reinterpret_cast<const float4*>(win + c * 4);
      float a = us[r][0] * w.x;
      a = fmaf(us[r][1], w.y, a);
      if (C > 2) a = fmaf(us[r][2], w.z, a);
      v = ZA0[n * ld + c] > 0.f ? a : 0.f;
    } else if (c < h + C) {
      v = us[r][c - h];
    } else {
      v = 0.f;
    }
    ZT0[n * ld + c] = v;
  }
}

// ------------------------------------------------------------------ tiled SGEMM with fused epilogues
struct GemmP {
  const float* A; const float* B; float* Cout;
  int64_t M; int N, K;
  int lda, ldb, ldc;
  int64_t sA, sB, sC;      // per-object strides
  const float* E0; int64_t sE0;  // fwd: previous ZA (copy aug columns); dgrad: previous ZA (relu mask)
  float* E1; int64_t sE1;        // dgrad: dX accumulate [N][4]
  int h, C;
  int64_t k_chunk;         // wgrad: pixel rows per split (blockIdx.x)
  int64_t sSplit;          // wgrad: stride between splits in Cout
  const float* Mz; int64_t sMz;  // tangent fwd: ZA_out of the forward (its relu mask)
};

// MODE 0: ZA_out = relu(ZA_in * Waug^T)                 A(m,k)=A[m*lda+k]   B(k,n)=B[n*ldb+k]
// MODE 1: delta_prev = (delta * Waug) .* (ZA_prev > 0)  A(m,k)=A[m*lda+k]   B(k,n)=B[k*ldb+n]
// MODE 2: dWaug[split] = delta^T * ZA_prev              A(m,k)=A[k*lda+m]   B(k,n)=B[k*ldb+n]
// MODE 3: ZT_out = (ZT_in * Waug^T) .* (ZA_out > 0)     as MODE 0: the tangent of MODE 0 along the tangent rows ZT_in
// A CTA writes a tile of kGemmTile output columns (and, in MODE 2, of kGemmTile output rows) chosen by blockIdx.y:
// rows wider than one tile (ld > 144, from h = 141) take several CTAs.  MODE 2 folds its row and column tiles into
// blockIdx.y (row tile major); blockIdx.x is the pixel block / split and blockIdx.z the object in every mode.
constexpr int kGemmTile = 144;

template <int MODE>
__global__ void __launch_bounds__(256) k_gemm(GemmP p) {
  constexpr int BM = (MODE == 2) ? kGemmTile : 128;
  constexpr int TM = BM / 16;
  constexpr int BN = kGemmTile, TN = 9, BK = 8;
  constexpr int NA = (BM * BK + 255) / 256, NB = (BN * BK + 255) / 256;
  __shared__ float As[2][BK][BM + 4];
  __shared__ float Bs[2][BK][BN + 4];

  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int o = blockIdx.z;
  const float* A = p.A + (int64_t)o * p.sA;
  const float* B = p.B + (int64_t)o * p.sB;
  int64_t m0 = 0, k_begin = 0, k_end = p.K;   // m0: first pixel row (modes 0, 1, 3) or first weight row (mode 2)
  int n0 = (int)blockIdx.y * BN;              // first output column
  if (MODE == 2) {
    const int col_tiles = (p.N + BN - 1) / BN;
    const int mt = (int)blockIdx.y / col_tiles;
    m0 = (int64_t)mt * BM;
    n0 = ((int)blockIdx.y - mt * col_tiles) * BN;
    k_begin = (int64_t)blockIdx.x * p.k_chunk;
    k_end = k_begin + p.k_chunk < p.K ? k_begin + p.k_chunk : (int64_t)p.K;
    if (k_end < k_begin) k_end = k_begin;
  } else {
    m0 = (int64_t)blockIdx.x * BM;
  }
  // operands and outputs seen from the tile's first column (and, in mode 2, first weight row): the loops below index them
  // as the single-tile kernel does, against limits shifted by the offset
  const int n_lim = ((MODE == 0 || MODE == 3) ? p.N : p.ldb) - n0;    // valid B columns of the tile
  B += (MODE == 0 || MODE == 3) ? (int64_t)n0 * p.ldb : (int64_t)n0;
  const int a_lim = p.lda - (MODE == 2 ? (int)m0 : 0);               // mode 2: valid A columns of the tile
  if (MODE == 2) A += m0;

  float ra[NA], rb[NB];
  auto gload = [&](int64_t k0) {
#pragma unroll
    for (int i = 0; i < NA; i++) {
      int e = tid + 256 * i;
      float v = 0.f;
      if (e < BM * BK) {
        if (MODE == 2) {  // m contiguous in global
          int k = e / BM, m = e - k * BM;
          int64_t kk = k0 + k;
          if (kk < k_end && m < a_lim) v = A[kk * p.lda + m];
        } else {          // k contiguous in global
          int m = e / BK, k = e - m * BK;
          int64_t kk = k0 + k;
          if (m0 + m < p.M && kk < p.lda) v = A[(m0 + m) * p.lda + kk];
        }
      }
      ra[i] = v;
    }
#pragma unroll
    for (int i = 0; i < NB; i++) {
      int e = tid + 256 * i;
      float v = 0.f;
      if (e < BN * BK) {
        if (MODE == 0 || MODE == 3) {  // k contiguous in global: B(k,n) = W[n][k], rows n < h
          int n = e / BK, k = e - n * BK;
          int64_t kk = k0 + k;
          if (n < n_lim && kk < p.ldb) v = B[(int64_t)n * p.ldb + kk];
        } else {          // n contiguous in global
          int k = e / BN, n = e - k * BN;
          int64_t kk = k0 + k;
          bool ok = (MODE == 1) ? (kk < p.K) : (kk < k_end);
          if (ok && n < n_lim) v = B[kk * p.ldb + n];
        }
      }
      rb[i] = v;
    }
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int i = 0; i < NA; i++) {
      int e = tid + 256 * i;
      if (e < BM * BK) {
        if (MODE == 2) { int k = e / BM, m = e - k * BM; As[buf][k][m] = ra[i]; }
        else { int m = e / BK, k = e - m * BK; As[buf][k][m] = ra[i]; }
      }
    }
#pragma unroll
    for (int i = 0; i < NB; i++) {
      int e = tid + 256 * i;
      if (e < BN * BK) {
        if (MODE == 0 || MODE == 3) { int n = e / BK, k = e - n * BK; Bs[buf][k][n] = rb[i]; }
        else { int k = e / BN, n = e - k * BN; Bs[buf][k][n] = rb[i]; }
      }
    }
  };

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; i++)
#pragma unroll
    for (int j = 0; j < TN; j++) acc[i][j] = 0.f;

  // K extent actually walked (operands are zero padded / guarded up to a multiple of BK)
  int64_t kw_end = (MODE == 2) ? k_end : (int64_t)((p.K + BK - 1) / BK * BK);
  int buf = 0;
  if (k_begin < kw_end) {
    gload(k_begin);
    sstore(0);
  }
  __syncthreads();
  for (int64_t k0 = k_begin; k0 < kw_end; k0 += BK) {
    bool more = k0 + BK < kw_end;
    if (more) gload(k0 + BK);
#pragma unroll
    for (int k = 0; k < BK; k++) {
      float a[TM], b[TN];
#pragma unroll
      for (int i = 0; i < TM; i++) a[i] = As[buf][k][ty + 16 * i];
#pragma unroll
      for (int j = 0; j < TN; j++) b[j] = Bs[buf][k][tx + 16 * j];
#pragma unroll
      for (int i = 0; i < TM; i++)
#pragma unroll
        for (int j = 0; j < TN; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (more) sstore(buf ^ 1);
    __syncthreads();
    buf ^= 1;
  }

  // ---- epilogue (column n of the tile is output column n0 + n)
  const int c_lim = p.ldc - n0, h_lim = p.h - n0;
  if (MODE == 0 || MODE == 3) {
    float* Cz = p.Cout + (int64_t)o * p.sC + n0;
    const float* Zin = p.E0 + (int64_t)o * p.sE0 + n0;
    const float* Zm = MODE == 3 ? p.Mz + (int64_t)o * p.sMz + n0 : nullptr;
#pragma unroll
    for (int i = 0; i < TM; i++) {
      int64_t m = m0 + ty + 16 * i;
      if (m >= p.M) continue;
#pragma unroll
      for (int j = 0; j < TN; j++) {
        int n = tx + 16 * j;
        if (n >= c_lim) continue;
        float v;
        if (MODE == 0) v = (n < h_lim) ? fmaxf(acc[i][j], 0.f) : Zin[m * p.ldc + n];
        else v = (n < h_lim) ? (Zm[m * p.ldc + n] > 0.f ? acc[i][j] : 0.f) : Zin[m * p.ldc + n];
        Cz[m * p.ldc + n] = v;
      }
    }
  } else if (MODE == 1) {
    float* Cd = p.Cout + (int64_t)o * p.sC + n0;
    const float* Zp = p.E0 + (int64_t)o * p.sE0 + n0;
    float* dX = p.E1 ? p.E1 + (int64_t)o * p.sE1 : nullptr;
#pragma unroll
    for (int i = 0; i < TM; i++) {
      int64_t m = m0 + ty + 16 * i;
      if (m >= p.M) continue;
#pragma unroll
      for (int j = 0; j < TN; j++) {
        int n = tx + 16 * j;
        if (n >= c_lim) continue;
        float v = 0.f;
        if (n < h_lim) {
          v = Zp[m * p.ldc + n] > 0.f ? acc[i][j] : 0.f;
        } else if (dX && n < h_lim + p.C) {
          dX[m * 4 + (n - h_lim)] += acc[i][j];   // one thread per (m, n): no race
        }
        Cd[m * p.ldc + n] = v;
      }
    }
  } else {
    float* Cw = p.Cout + (int64_t)blockIdx.x * p.sSplit + (int64_t)o * p.sC + m0 * p.ldc + n0;
    const int m_lim = p.h - (int)m0;
#pragma unroll
    for (int i = 0; i < TM; i++) {
      int m = ty + 16 * i;
      if (m >= m_lim) continue;
#pragma unroll
      for (int j = 0; j < TN; j++) {
        int n = tx + 16 * j;
        if (n >= c_lim) continue;
        Cw[(int64_t)m * p.ldc + n] = acc[i][j];
      }
    }
  }
}

// ------------------------------------------------------------------ output layer + loss (a7 last line, a9, a10)
struct OutP {
  const float* ZA; int64_t sZA;   // ZA_L
  const float* waug; int64_t G, aug_out;
  float* logits;                  // [O][N]
  // training
  int train;                      // 0 forward only, 1 loss-driven (fit), 2 upstream dlogits
  const float* target;            // [O][N]
  const float* dlogits;           // [O][N]
  LossCoef loss[16];
  float* D; int64_t sD;           // delta_L out
  float* dX; int64_t sdX;         // optional: coordinate gradient init
  float* part; int64_t sSplit;    // partial sums [S][O][G]
  float* lossp;                   // [S][O]
  int64_t N, chunk;
  int h, C, ld, O;
  LossPix pix[16];                // WL: weight map and ignore label per object
};

// WL: the loss carries per-pixel weights and / or an ignore label (awb_loss_spec); the other instantiation is the plain
// loss and does not read pix
template <int Q, bool WL>
__global__ void __launch_bounds__(256) k_out(OutP p) {
  extern __shared__ float sm[];   // [8][ld] gradient partials + [8] loss
  const int s = blockIdx.x, o = blockIdx.y;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* wo = p.waug + (int64_t)o * p.G + p.aug_out;
  const float* Z = p.ZA + (int64_t)o * p.sZA;
  float wq[Q], gacc[Q];
#pragma unroll
  for (int q = 0; q < Q; q++) {
    int c = lane + 32 * q;
    wq[q] = c < p.ld ? wo[c] : 0.f;
    gacc[q] = 0.f;
  }
  float lacc = 0.f;
  int64_t r0 = (int64_t)s * p.chunk;
  int64_t r1 = r0 + p.chunk < p.N ? r0 + p.chunk : p.N;
  LossCoef ls = p.loss[p.train == 1 ? o : 0];
  const LossPix lp = p.pix[WL ? o : 0];
  for (int64_t n = r0 + w; n < r1; n += 8) {
    float z[Q];
    float dot = 0.f;
#pragma unroll
    for (int q = 0; q < Q; q++) {
      int c = lane + 32 * q;
      z[q] = c < p.ld ? Z[n * p.ld + c] : 0.f;
      dot = fmaf(z[q], wq[q], dot);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, off);
    float y = dot;
    if (lane == 0 && p.logits) p.logits[(int64_t)o * p.N + n] = y;
    if (p.train == 0) continue;
    float dy;
    if (p.train == 1) {
      float t = p.target[(int64_t)o * p.N + n];
      bool fg = ls.cls_rule == AWB_CLS_UNARY_LT_HALF ? (t < 0.5f) : (t != 1.0f);
      float coef = fg ? ls.coef_fg : ls.coef_bg;
      if (WL && lp.weight) coef *= lp.weight[(int64_t)n];   // w * coef: a weight of 1 leaves every bit of the loss
      float sg = 1.f / (1.f + expf(-y));
      float l;
      if (ls.kind == AWB_LOSS_SE_SIGMOID) {
        float d = t - sg;
        l = d * d;
        dy = coef * (-2.f * d) * sg * (1.f - sg);
      } else {
        l = fmaxf(y, 0.f) - y * t + log1pf(expf(-fabsf(y)));
        dy = coef * (sg - t);
      }
      if (WL) {   // select, do not multiply: a NaN logit, target or weight of an ignored pixel cannot leak in
        const bool keep = loss_keep(lp, t);
        dy = keep ? dy : 0.f;
        lacc = fmaf(keep ? coef : 0.f, keep ? l : 0.f, lacc);   // the contraction of the plain loss's lacc += coef * l
      } else {
        lacc += coef * l;
      }
    } else {
      dy = p.dlogits[(int64_t)o * p.N + n];
    }
    float* Dr = p.D + (int64_t)o * p.sD + n * p.ld;
#pragma unroll
    for (int q = 0; q < Q; q++) {
      int c = lane + 32 * q;
      if (c < p.ld) {
        Dr[c] = (c < p.h && z[q] > 0.f) ? dy * wq[q] : 0.f;
        gacc[q] = fmaf(dy, z[q], gacc[q]);
      }
    }
    if (p.dX && lane < 4) {
      // d y / d x = s_o  (out.skp.weight); columns h .. h+C-1 of waug_out
      float so = (lane < p.C) ? wo[p.h + lane] : 0.f;
      p.dX[(int64_t)o * p.sdX + n * 4 + lane] = dy * so;
    }
  }
  // block reduce: fixed order over the 8 warps
  float* gs = sm;
  float* lsum = sm + 8 * p.ld;
#pragma unroll
  for (int q = 0; q < Q; q++) {
    int c = lane + 32 * q;
    if (c < p.ld) gs[w * p.ld + c] = gacc[q];
  }
  if (lane == 0) lsum[w] = lacc;   // all lanes of a warp hold identical lacc
  __syncthreads();
  if (p.train != 0) {
    for (int c = threadIdx.x; c < p.ld; c += 256) {
      float a = 0.f;
#pragma unroll
      for (int ww = 0; ww < 8; ww++) a += gs[ww * p.ld + c];
      p.part[(int64_t)s * p.sSplit + (int64_t)o * p.G + p.aug_out + c] = a;
    }
    if (threadIdx.x == 0) {
      float a = 0.f;
#pragma unroll
      for (int ww = 0; ww < 8; ww++) a += lsum[ww];
      p.lossp[s * p.O + o] = a;
    }
  }
}

// ------------------------------------------------------------------ tangent output layer (second-order pass)
// Per pixel: ydot = waug_out . ZT_L (= w_o . zdot_L + s_o . u, the derivative of the logit along u), written to ydot[n];
// delta_L = w .* w_o .* (z_L > 0) exactly as k_out seeds it from dlogits = w; the output layer's partials sum w * ZT_L
// (d w_o = sum w zdot_L, d s_o = sum w u, d b_o = 0).  Single object; pixel range s = blockIdx.x, fixed-order block sum.
struct TanOutP {
  const float* ZA;                // ZA_L (relu mask)
  const float* ZT;                // ZT_L
  const float* waug; int64_t aug_out;
  const float* w;                 // [N] dlogits of the first backward
  float* ydot;                    // [N]
  float* D;                       // delta_L out
  float* part; int64_t sSplit;    // partial sums [S][G]
  int64_t N, chunk;
  int h, ld;
};

template <int Q>
__global__ void __launch_bounds__(256) k_tan_out(TanOutP p) {
  extern __shared__ float sm[];   // [8][ld] gradient partials
  const int s = blockIdx.x;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* wo = p.waug + p.aug_out;
  float wq[Q], gacc[Q];
#pragma unroll
  for (int q = 0; q < Q; q++) {
    int c = lane + 32 * q;
    wq[q] = c < p.ld ? wo[c] : 0.f;
    gacc[q] = 0.f;
  }
  int64_t r0 = (int64_t)s * p.chunk;
  int64_t r1 = r0 + p.chunk < p.N ? r0 + p.chunk : p.N;
  for (int64_t n = r0 + w; n < r1; n += 8) {
    float zt[Q];
    float dot = 0.f;
#pragma unroll
    for (int q = 0; q < Q; q++) {
      int c = lane + 32 * q;
      zt[q] = c < p.ld ? p.ZT[n * p.ld + c] : 0.f;
      dot = fmaf(zt[q], wq[q], dot);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, off);
    if (lane == 0) p.ydot[n] = dot;
    const float dy = p.w[n];
    float* Dr = p.D + n * p.ld;
#pragma unroll
    for (int q = 0; q < Q; q++) {
      int c = lane + 32 * q;
      if (c < p.ld) {
        Dr[c] = (c < p.h && p.ZA[n * p.ld + c] > 0.f) ? dy * wq[q] : 0.f;
        gacc[q] = fmaf(dy, zt[q], gacc[q]);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < Q; q++) {
    int c = lane + 32 * q;
    if (c < p.ld) sm[w * p.ld + c] = gacc[q];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < p.ld; c += 256) {
    float a = 0.f;
#pragma unroll
    for (int ww = 0; ww < 8; ww++) a += sm[ww * p.ld + c];
    p.part[(int64_t)s * p.sSplit + p.aug_out + c] = a;
  }
}

// ------------------------------------------------------------------ input layer backward
// dW_in[j][c] = sum_n delta0[n][j] x[n][c];  db_in[j] = sum_n delta0[n][j] one  (one = 1; 0 against tangent rows,
// whose bias input is the tangent of a constant: fmaf(d, 1, a) rounds like a + d, so the first-order bits are kept)
__global__ void __launch_bounds__(256) k_in_wgrad(const float* __restrict__ D0, int64_t sD,
                                                  const float* __restrict__ X, float* __restrict__ part,
                                                  int64_t sSplit, int64_t G, int64_t aug_in, int64_t N,
                                                  int64_t chunk, int h, int ld, float one) {
  int s = blockIdx.x, o = blockIdx.y, j = threadIdx.x;
  const float* D = D0 + (int64_t)o * sD;
  const float* Xo = X + (int64_t)o * N * 4;
  int64_t r0 = (int64_t)s * chunk, r1 = r0 + chunk < N ? r0 + chunk : N;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  if (j < h) {
    for (int64_t n = r0; n < r1; n++) {
      float d = D[n * ld + j];
      float4 x = *reinterpret_cast<const float4*>(Xo + n * 4);
      a0 = fmaf(d, x.x, a0); a1 = fmaf(d, x.y, a1); a2 = fmaf(d, x.z, a2); a3 = fmaf(d, one, a3);
    }
    float* out = part + (int64_t)s * sSplit + (int64_t)o * G + aug_in + j * 4;
    *reinterpret_cast<float4*>(out) = make_float4(a0, a1, a2, a3);
  }
}

// dX[n][c] += sum_j delta0[n][j] W_in[j][c]   (only when the coordinates need a gradient)
__global__ void __launch_bounds__(256) k_in_dgrad(const float* __restrict__ D0, int64_t sD,
                                                  const float* __restrict__ waug, int64_t G, int64_t aug_in,
                                                  float* __restrict__ dX, int64_t N, int h, int ld) {
  int o = blockIdx.y;
  int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int64_t n = (int64_t)blockIdx.x * 8 + w;
  if (n >= N) return;
  const float* D = D0 + (int64_t)o * sD + n * ld;
  const float* win = waug + (int64_t)o * G + aug_in;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f;
  for (int j = lane; j < h; j += 32) {
    float d = D[j];
    float4 wv = *reinterpret_cast<const float4*>(win + j * 4);
    a0 = fmaf(d, wv.x, a0); a1 = fmaf(d, wv.y, a1); a2 = fmaf(d, wv.z, a2);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    a0 += __shfl_xor_sync(0xffffffffu, a0, off);
    a1 += __shfl_xor_sync(0xffffffffu, a1, off);
    a2 += __shfl_xor_sync(0xffffffffu, a2, off);
  }
  if (lane == 0) {
    float* d = dX + ((int64_t)o * N + n) * 4;
    d[0] += a0; d[1] += a1; d[2] += a2;
  }
}

// ------------------------------------------------------------------ optimizer (a11) + clamp (a8) + plateau (K12)
// step_size = lr / (1 - beta1^t) and bc2s = sqrt(1 - beta2^t) are evaluated in double once per block
// (torch computes them as Python floats), see k_reduce_opt.
__device__ __forceinline__ void opt_update(int kind, float& p, float g, float& m, float& v, float step_size,
                                           float bc2s, float beta1, float beta2, float eps, float wd) {
  // torch/optim/adam.py::_single_tensor_adam, torch/optim/adamax.py::_single_tensor_adamax
  if (wd != 0.f) g = fmaf(wd, p, g);
  m = m + (g - m) * (1.f - beta1);                       // exp_avg.lerp_(grad, 1 - beta1)
  if (kind == AWB_OPT_ADAM) {
    v = v * beta2 + (1.f - beta2) * g * g;               // mul_(beta2).addcmul_(g, g, 1 - beta2)
    float denom = sqrtf(v) / bc2s + eps;
    p = p - step_size * (m / denom);
  } else {
    v = fmaxf(v * beta2, fabsf(g) + eps);                // exp_inf
    p = p - step_size * (m / v);
  }
}

struct OptP {
  float* params; float* m; float* v; OptScal* scal;
  const float* part; int64_t sSplit; int S;      // ICNN partials [S][O][G]
  const float* fpart; int64_t sFSplit; int SF;   // flow+linear partials [SF][O][PF]
  const float* lossp; int64_t sLoss;             // loss partial s of object o at lossp[s * sLoss + o]
  const float* grads;                            // direct gradients (awb_optim_step) or null
  const int32_t* map; const uint8_t* clamp; const uint8_t* group;
  int64_t P, off_icnn, P_icnn, off_flow, PF, G;
  int O;
  awb_opt_hyper hy;
  float* loss_out;
};

// Block = 32 consecutive parameters x 8 warps; warp w sums its fixed range of the <=148 per-CTA partials
// (coalesced 128-byte rows, independent loads in flight), the ranges are combined in a fixed order, then
// warp 0 applies Adam/Adamax + L2 + clamp.  The last block to finish (ticket in OptScal.pad) advances the
// step counter and the plateau scheduler, so a fit step needs no separate scheduler launch.
__global__ void __launch_bounds__(256) k_reduce_opt(OptP a, int n_groups, int use_loss) {
  __shared__ float s_loss;
  __shared__ float s_part[8][32];
  __shared__ float s_step_size[AWB_MAX_GROUPS], s_bc2s[AWB_MAX_GROUPS];
  const int o = blockIdx.y;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x >= 32 && threadIdx.x < 32 + AWB_MAX_GROUPS) {   // bias corrections, once per block and group
    const int g = threadIdx.x - 32;
    int step1 = a.scal[o].step + 1 - a.scal[o].group_start[g];
    if (step1 < 1) step1 = 1;
    const double bc1 = 1.0 - pow((double)a.hy.beta1, (double)step1);
    s_step_size[g] = (float)(a.scal[o].lr[g] / bc1);
    s_bc2s[g] = (float)sqrt(1.0 - pow((double)a.hy.beta2, (double)step1));
  }
  if (a.lossp) {
    if (w == 0) {
      // fixed-order loss sum: lane-strided then butterfly
      float l = 0.f;
      const int SL = a.S > 0 ? a.S : a.SF;
      for (int s = lane; s < SL; s += 32) l += a.lossp[s * a.sLoss + o];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) l += __shfl_xor_sync(0xffffffffu, l, off);
      if (lane == 0) s_loss = l;
    }
  }
  __syncthreads();
  // reference raises before backward() on a non-finite loss: leave the parameters untouched
  const bool bad = a.lossp && !isfinite(s_loss);
  const int64_t i = (int64_t)blockIdx.x * 32 + lane;
  const bool mine = i < a.P && !(a.hy.active_groups && !((a.hy.active_groups >> a.group[i]) & 1));
  if (!bad && !a.grads) {
    float g = 0.f;
    if (mine) {
      const float* src;
      int64_t stride;
      int S;
      if (i >= a.off_icnn && i < a.off_icnn + a.P_icnn) { src = a.part + (int64_t)o * a.G + a.map[i - a.off_icnn]; stride = a.sSplit; S = a.S; }
      else { src = a.fpart + (int64_t)o * a.PF + (i - a.off_flow); stride = a.sFSplit; S = a.SF; }
      const int s0 = (S * w) >> 3, s1 = (S * (w + 1)) >> 3;
#pragma unroll 4
      for (int s = s0; s < s1; s++) g += src[(int64_t)s * stride];
    }
    s_part[w][lane] = g;
    __syncthreads();
  }
  if (!bad && w == 0 && mine) {
    float g;
    if (a.grads) {
      g = a.grads[(int64_t)o * a.P + i];
    } else {
      g = 0.f;
#pragma unroll
      for (int ww = 0; ww < 8; ww++) g += s_part[ww][lane];
    }
    const int grp = a.group[i];
    const int64_t gi = (int64_t)o * a.P + i;
    float p = a.params[gi], m = a.m[gi], v = a.v[gi];
    opt_update(a.hy.kind, p, g, m, v, s_step_size[grp], s_bc2s[grp], a.hy.beta1, a.hy.beta2, a.hy.eps,
               a.hy.weight_decay[grp]);
    if (a.clamp[i]) p = fmaxf(p, 0.f);                     // enforce_convexity
    a.params[gi] = p; a.m[gi] = m; a.v[gi] = v;
  }
  // ---- ticket: the last block of this object closes the step (every block has read scal by then)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    OptScal& s = a.scal[o];
    const int t = atomicAdd(&s.pad, 1);
    if (t == (int)gridDim.x - 1) {
      s.pad = 0;
      if (a.lossp) { s.last_loss = s_loss; if (a.loss_out) a.loss_out[o] = s_loss; }
      if (bad) {
        s.nonfinite = 1;
      } else {
        // step counter + ReduceLROnPlateau.step(loss) (torch/optim/lr_scheduler.py)
        s.step += 1;
        if (a.hy.active_groups)
          for (int g = 0; g < AWB_MAX_GROUPS; g++)
            if (!((a.hy.active_groups >> g) & 1)) s.group_start[g] += 1;
        if (a.hy.plateau_enabled && use_loss) {
          const double cur = (double)s_loss;
          if (cur < s.best * (1.0 - (double)a.hy.threshold)) { s.best = cur; s.num_bad = 0; }
          else s.num_bad += 1;
          if (s.num_bad > a.hy.patience) {
            for (int g = 0; g < n_groups; g++) {
              double nl = s.lr[g] * (double)a.hy.factor;
              if (nl < (double)a.hy.min_lr) nl = (double)a.hy.min_lr;
              if (s.lr[g] - nl > (double)a.hy.plateau_eps) s.lr[g] = nl;
            }
            s.num_bad = 0;
          }
        }
      }
    }
  }
}

// ICNN priors: the same step in augmented-index space.  A block owns 128 consecutive augmented entries; warp w
// sums its fixed slice of the partials with coalesced float4 loads (all in flight at once), the slices are
// combined in a fixed order, and one thread per entry applies the optimizer through the inverse map.  With a
// tensor-path workspace the updated parameter is also written into the fp16 weight image of the next step.
struct OptA {
  float* params; float* m; float* v; OptScal* scal;
  const float* part; int64_t sSplit; int S;
  const float* lossp;
  const int32_t* imap; const uint8_t* clamp; const uint8_t* group;
  int64_t P, off_icnn, G, aug_out;
  int O, ld;
  awb_opt_hyper hy;
  float* loss_out;
  uint8_t* img; int64_t img_stride, vec_off; const int32_t* aug2img;
  // flow priors: blocks nb_aug .. gridDim.x - 1 own 128 consecutive flow / linear parameters each (state_dict order)
  const float* fpart; int64_t sFSplit, off_flow, PF; int SF, nb_aug;
};

__global__ void __launch_bounds__(256) k_reduce_opt_aug(OptA a, int n_groups) {
  __shared__ float s_loss;
  __shared__ float4 s_part[8][32];
  __shared__ float s_step_size[AWB_MAX_GROUPS], s_bc2s[AWB_MAX_GROUPS];
  const int o = blockIdx.y;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t g0 = (int64_t)blockIdx.x * 128;
  // ---- before the producer of the partials has finished (programmatic dependent launch: these blocks become
  // resident as the fit kernel's CTAs retire): everything that only depends on the previous optimizer step --
  // bias corrections, index maps, the parameter and its moments.
  if (threadIdx.x >= 128 && threadIdx.x < 128 + AWB_MAX_GROUPS) {   // bias corrections, once per block and group
    const int g = threadIdx.x - 128;
    int step1 = a.scal[o].step + 1 - a.scal[o].group_start[g];      // the group's own step count, as in k_reduce_opt
    if (step1 < 1) step1 = 1;
    const double bc1 = 1.0 - pow((double)a.hy.beta1, (double)step1);
    s_step_size[g] = (float)(a.scal[o].lr[g] / bc1);
    s_bc2s[g] = (float)sqrt(1.0 - pow((double)a.hy.beta2, (double)step1));
  }
  const int t = threadIdx.x;
  const bool flow_blk = (int)blockIdx.x >= a.nb_aug && a.nb_aug > 0;
  const int64_t fj0 = flow_blk ? ((int64_t)blockIdx.x - a.nb_aug) * 128 : 0;     // first flow / linear parameter of the block
  const int64_t aug = g0 + t;
  int64_t gi = -1;
  int grp = 0, e = -1;
  bool do_clamp = false;
  float p = 0.f, m = 0.f, v = 0.f;
  if (flow_blk) {
    if (t < 128 && fj0 + t < a.PF) {
      const int64_t i = a.off_flow + fj0 + t;
      grp = a.group[i];
      if (!(a.hy.active_groups && !((a.hy.active_groups >> grp) & 1))) {
        gi = (int64_t)o * a.P + i;
        p = a.params[gi]; m = a.m[gi]; v = a.v[gi];
      }
    }
  } else if (t < 128 && aug < a.G) {
    const int32_t li = a.imap[aug];
    if (li >= 0) {
      const int64_t i = a.off_icnn + li;
      grp = a.group[i];
      if (!(a.hy.active_groups && !((a.hy.active_groups >> grp) & 1))) {
        gi = (int64_t)o * a.P + i;
        do_clamp = a.clamp[i] != 0;
        p = a.params[gi]; m = a.m[gi]; v = a.v[gi];
        if (a.img) e = a.aug2img[aug];
      }
    }
  }
  grid_dep_wait();      // the partials and the loss sums are complete
  grid_dep_launch();
  // every warp's partial rows and warp 0's loss terms go out together: one L2 round trip and one barrier between the
  // end of the fit kernel and the parameter update (this stretch is not hidden by anything)
  float lsum = 0.f;
  if (w == 0)
    for (int s = lane; s < a.S; s += 32) lsum += __ldcg(a.lossp + s * a.O + o);
  if (flow_blk) {
    // flow / linear partials [SF][O][PF]: lane owns columns lane + 32 k of the block (rows need not be 16-byte aligned)
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    const float* src = a.fpart + (int64_t)o * a.PF + fj0;
    const int s0 = (a.SF * w) >> 3, s1 = (a.SF * (w + 1)) >> 3;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if (fj0 + lane + 32 * k < a.PF) {
#pragma unroll 4
        for (int sb = s0; sb < s1; sb++) acc[k] += __ldcg(src + (int64_t)sb * a.sFSplit + lane + 32 * k);
      }
    }
#pragma unroll
    for (int k = 0; k < 4; k++) reinterpret_cast<float*>(&s_part[w][0])[lane + 32 * k] = acc[k];
  } else {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (g0 + 4 * lane < a.G) {
      const float4* src = reinterpret_cast<const float4*>(a.part + (int64_t)o * a.G + g0) + lane;
      const int64_t stride4 = a.sSplit / 4;
      const int s0 = (a.S * w) >> 3, s1 = (a.S * (w + 1)) >> 3;
      // all of this warp's <= 19 partial rows in flight at once, summed in a fixed order
      for (int sb = s0; sb < s1; sb += 20) {
        float4 tt[20];
#pragma unroll
        for (int k = 0; k < 20; k++)
          tt[k] = sb + k < s1 ? __ldcg(src + (int64_t)(sb + k) * stride4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < 20; k++) { acc.x += tt[k].x; acc.y += tt[k].y; acc.z += tt[k].z; acc.w += tt[k].w; }
      }
    }
    s_part[w][lane] = acc;
  }
  if (w == 0) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, off);
    if (lane == 0) s_loss = lsum;
  }
  __syncthreads();
  const bool bad = !isfinite(s_loss);
  if (!bad) {
    if (gi >= 0) {
      float g = 0.f;
#pragma unroll
      for (int ww = 0; ww < 8; ww++) g += reinterpret_cast<const float*>(&s_part[ww][0])[t];
      opt_update(a.hy.kind, p, g, m, v, s_step_size[grp], s_bc2s[grp], a.hy.beta1, a.hy.beta2, a.hy.eps,
                 a.hy.weight_decay[grp]);
      if (do_clamp) p = fmaxf(p, 0.f);                     // enforce_convexity
      a.params[gi] = p; a.m[gi] = m; a.v[gi] = v;
      if (a.img) {   // keep the tensor path's fp16 weight image in step
        uint8_t* base = a.img + (int64_t)o * a.img_stride;
        if (e >= 0) reinterpret_cast<__half*>(base)[e] = __float2half_rn(p);
        if (!flow_blk && aug >= a.aug_out) {
          const int k = (int)(aug - a.aug_out);
          reinterpret_cast<float*>(base + a.vec_off)[k] = p;
          reinterpret_cast<__half*>(base + a.vec_off + 4 * 144)[k] = __float2half_rn(p);
        }
      }
    }
  }
  // ---- ticket: the last block of this object closes the step (every block has read scal by then)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    OptScal& s = a.scal[o];
    const int t = atomicAdd(&s.pad, 1);
    if (t == (int)gridDim.x - 1) {
      s.pad = 0;
      s.last_loss = s_loss;
      if (a.loss_out) a.loss_out[o] = s_loss;
      if (bad) {
        s.nonfinite = 1;
      } else {
        s.step += 1;
        if (a.hy.active_groups)
          for (int g = 0; g < AWB_MAX_GROUPS; g++)
            if (!((a.hy.active_groups >> g) & 1)) s.group_start[g] += 1;
        if (a.hy.plateau_enabled) {
          const double cur = (double)s_loss;
          if (cur < s.best * (1.0 - (double)a.hy.threshold)) { s.best = cur; s.num_bad = 0; }
          else s.num_bad += 1;
          if (s.num_bad > a.hy.patience) {
            for (int g = 0; g < n_groups; g++) {
              double nl = s.lr[g] * (double)a.hy.factor;
              if (nl < (double)a.hy.min_lr) nl = (double)a.hy.min_lr;
              if (s.lr[g] - nl > (double)a.hy.plateau_eps) s.lr[g] = nl;
            }
            s.num_bad = 0;
          }
        }
      }
    }
  }
}

__global__ void k_absmax(const float* __restrict__ x, int64_t n, float* out) {
  const int o = blockIdx.x;
  const float* p = x + (int64_t)o * n;
  float m = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, fabsf(p[i]));
  __shared__ float red[32];
  for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 0; i < (int)(blockDim.x >> 5); i++) m = fmaxf(m, red[i]);
    out[o] = m;
  }
}

// max |w[i]| over the kept pixels of object blockIdx.y, grid-stride over blockIdx.x, combined with an integer atomicMax on
// the bits of a non-negative float (fmaxf drops a NaN weight; a kept NaN weight makes the loss itself non-finite)
struct WAbsP {
  LossPix pix[16];
  const float* t;   // [O][n]
  int64_t n;
  float* out;       // [O], zeroed
};
__global__ void __launch_bounds__(256) k_weight_absmax(WAbsP p) {
  const int o = blockIdx.y;
  const LossPix pix = p.pix[o];
  const float* t = p.t + (int64_t)o * p.n;
  float m = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < p.n; i += (int64_t)gridDim.x * 256)
    if (loss_keep(pix, t[i])) m = fmaxf(m, pix.weight ? fabsf(pix.weight[i]) : 1.f);
  for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(p.out + o), __float_as_int(m));
}

int weight_absmax_per_object(const awb_loss_spec* loss, const float* target, int64_t n, int O, float* out,
                             cudaStream_t st) {
  AWB_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * O, st));
  WAbsP p = {};
  for (int o = 0; o < O && o < 16; o++) p.pix[o] = loss_pix(loss[o]);
  p.t = target; p.n = n; p.out = out;
  const int per_obj = kMaxSplits / O > 0 ? kMaxSplits / O : 1;
  const int blocks = (int)((n + 2047) / 2048 < per_obj ? (n + 2047) / 2048 : per_obj);
  AWB_LAUNCH(PK_MISC, st, k_weight_absmax<<<dim3(blocks, O), 256, 0, st>>>(p));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int absmax_per_object(const float* x, int64_t n, int O, float* out, cudaStream_t st) {
  AWB_LAUNCH(PK_MISC, st, k_absmax<<<O, 1024, 0, st>>>(x, n, out));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

// grads[o][i] = sum of the partials of parameter i in fixed partial order.  loss_slot (single object): thread P writes the
// sum of the S loss partials behind the gradient -- the [P + 1] gradient row of awb_prior_slice_grads.
__global__ void k_reduce_grads(float* grads, const float* part, int64_t sSplit, int S, int SF, const float* fpart,
                               int64_t sFSplit, const int32_t* map, int64_t P, int64_t off_icnn,
                               int64_t P_icnn, int64_t off_flow, int64_t PF, int64_t G, const float* lossp,
                               float* loss_slot) {
  grid_dep_wait();      // the partials are complete
  grid_dep_launch();
  int o = blockIdx.y;
  int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (loss_slot && i == P) {
    float l = 0.f;
    for (int s = 0; s < S; s++) l += lossp[s];
    *loss_slot = l;
    return;
  }
  if (i >= P) return;
  float g = 0.f;
  if (i >= off_icnn && i < off_icnn + P_icnn) {
    const float* src = part + (int64_t)o * G + map[i - off_icnn];
    for (int s = 0; s < S; s++) g += src[(int64_t)s * sSplit];
  } else {
    const float* src = fpart + (int64_t)o * PF + (i - off_flow);
    for (int s = 0; s < SF; s++) g += src[(int64_t)s * sFSplit];
  }
  grads[(int64_t)o * P + i] = g;
}

__global__ void k_clamp(float* params, const uint8_t* clamp, int64_t P) {
  int o = blockIdx.y;
  int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i < P && clamp[i]) { float& p = params[(int64_t)o * P + i]; p = fmaxf(p, 0.f); }
}

__global__ void k_opt_init(OptScal* scal, double l0, double l1, double l2, double l3, int O) {
  int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= O) return;
  OptScal s;
  s.lr[0] = l0; s.lr[1] = l1; s.lr[2] = l2; s.lr[3] = l3;
  s.best = INFINITY; s.step = 0; s.num_bad = 0; s.nonfinite = 0; s.pad = 0; s.last_loss = 0.f; s.pad2 = 0.f;
  for (int g = 0; g < AWB_MAX_GROUPS; g++) s.group_start[g] = 0;
  scal[o] = s;
}

__global__ void k_opt_set_lr(OptScal* scal, double l0, double l1, double l2, double l3, int O) {
  int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= O) return;
  scal[o].lr[0] = l0; scal[o].lr[1] = l1; scal[o].lr[2] = l2; scal[o].lr[3] = l3;
}

// dgrid[b][c][i][j] = dX[n][c]   (planar reference layout)
__global__ void k_dgrid(const float* dX, float* dgrid, int64_t N, int64_t HW, int C) {
  int64_t n = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (n >= N) return;
  int64_t b = n / HW, r = n - b * HW;
  for (int c = 0; c < C; c++) dgrid[(b * C + c) * HW + r] = dX[n * 4 + c];
}

// dX[n] = (d_deformed[n][0..C), 0...): a caller gradient on the deformed coordinates, in the layout the flow backward reads
__global__ void k_seed_dX(const float* dd, float* dX, int64_t N, int C) {
  int64_t n = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (n >= N) return;
  float d[3] = {0.f, 0.f, 0.f};
  for (int c = 0; c < C; c++) d[c] = dd[n * C + c];
  *reinterpret_cast<float4*>(dX + n * 4) = make_float4(d[0], d[1], d[2], 0.f);
}

// ======================================================================= host launchers
static GridDev to_dev(const awb_grid_spec* g, int C, int64_t row0) {
  GridDev d;
  d.mode = g->mode; d.B = g->B; d.H = g->H; d.W = g->W; d.C = C;
  d.t0 = g->t0; d.t_step = g->t_step; d.grid = g->grid; d.row0 = (uint32_t)row0;
  return d;
}

// k_gemm's blockIdx.y extent: column tiles over ld (modes 0, 1, 3); row tiles over h times column tiles (mode 2)
static unsigned gemm_col_tiles(const Layout& L) { return (unsigned)((L.ld + kGemmTile - 1) / kGemmTile); }
static unsigned gemm_wgrad_tiles(const Layout& L) { return (unsigned)((L.h + kGemmTile - 1) / kGemmTile) * gemm_col_tiles(L); }

static void opt_ptrs(const awb_prior* h, void* opt_state, float** m, float** v, OptScal** sc) {
  int64_t n = h->lay.P * h->desc.n_objects;
  *m = (float*)opt_state;
  *v = *m + n;
  *sc = (OptScal*)((char*)opt_state + round_up(2 * n * 4, 256));
}

int simt_forward(const awb_prior* h, const float* params, const awb_grid_spec* g, float* logits_out, bool training,
                 bool x_ready, const Workspace& ws, cudaStream_t st) {
  const Layout& L = h->lay;
  const int O = h->desc.n_objects;
  const int64_t N = ws.N;
  AWB_CUDA(cudaMemsetAsync(ws.waug, 0, sizeof(float) * O * L.G, st));
  AWB_LAUNCH(PK_PACK, st, k_pack<<<dim3((unsigned)((L.P_icnn + 255) / 256), O), 256, 0, st>>>(params, ws.waug, h->d_map, (int)L.P_icnn,
                                                                       L.P, L.off_icnn, L.G));
  const int64_t sLayer = N * L.ld;            // one ZA layer
  const int64_t sZAobj = (L.L + 1) * sLayer;  // all layers of an object
  AWB_LAUNCH(PK_INPUT, st, k_input<<<dim3((unsigned)((N + 63) / 64), O), 256, 0, st>>>(to_dev(g, L.C, ws.row0), (int)x_ready, ws.X, ws.waug, ws.ZA, N,
                                                              L.h, L.C, L.ld, L.G, L.aug_in, sZAobj));
  for (int i = 0; i < L.L; i++) {
    GemmP p = {};
    p.A = ws.ZA + i * sLayer; p.sA = sZAobj; p.lda = L.ld;
    p.B = ws.waug + L.aug_layer + (int64_t)i * L.h * L.ld; p.sB = L.G; p.ldb = L.ld;
    p.Cout = ws.ZA + (i + 1) * sLayer; p.sC = sZAobj; p.ldc = L.ld;
    p.M = N; p.N = L.h; p.K = L.ld;
    p.E0 = p.A; p.sE0 = sZAobj;
    p.h = L.h; p.C = L.C;
    AWB_LAUNCH(PK_GEMM_FWD, st, k_gemm<0><<<dim3((unsigned)((N + 127) / 128), gemm_col_tiles(L), O), 256, 0, st>>>(p));
  }
  if (!training || logits_out) {   // a training forward without logits leaves k_out to the backward
    OutP q = {};
    q.ZA = ws.ZA + L.L * sLayer; q.sZA = sZAobj;
    q.waug = ws.waug; q.G = L.G; q.aug_out = L.aug_out;
    q.logits = logits_out; q.train = 0; q.N = N; q.chunk = split_chunk(N);
    q.h = L.h; q.C = L.C; q.ld = L.ld; q.O = O;
    size_t smem = (8 * L.ld + 8) * sizeof(float);
    if (L.ld <= 160) AWB_LAUNCH(PK_OUT_LOSS, st, k_out<5, false><<<dim3(n_splits(N), O), 256, smem, st>>>(q));
    else AWB_LAUNCH(PK_OUT_LOSS, st, k_out<9, false><<<dim3(n_splits(N), O), 256, smem, st>>>(q));
  }
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int simt_backward(const awb_prior* h, const float* target, const awb_loss_spec* loss, const float* dlogits, bool need_dx,
                  const Workspace& ws, cudaStream_t st) {
  const Layout& L = h->lay;
  const int O = h->desc.n_objects;
  const int64_t N = ws.N;
  const int S = n_splits(N);
  const int64_t chunk = split_chunk(N);
  const int64_t sLayer = N * L.ld, sZAobj = (L.L + 1) * sLayer, sDobj = 2 * sLayer;
  const int64_t sSplit = (int64_t)O * L.G;

  OutP q = {};
  q.ZA = ws.ZA + L.L * sLayer; q.sZA = sZAobj;
  q.waug = ws.waug; q.G = L.G; q.aug_out = L.aug_out;
  q.logits = loss ? ws.logits : nullptr;
  q.train = loss ? 1 : 2;
  q.target = target; q.dlogits = dlogits;
  bool wl = false;
  if (loss)
    for (int o = 0; o < O && o < 16; o++) {
      q.loss[o] = loss_coef(loss[o]);
      q.pix[o] = loss_pix(loss[o]);
      wl = wl || loss_is_weighted(loss[o]);
    }
  q.D = ws.D + (L.L & 1) * sLayer; q.sD = sDobj;      // delta_i lives in D[i & 1]
  q.dX = need_dx ? ws.dX : nullptr; q.sdX = N * 4;
  q.part = ws.part; q.sSplit = sSplit; q.lossp = ws.lossp;
  q.N = N; q.chunk = chunk; q.h = L.h; q.C = L.C; q.ld = L.ld; q.O = O;
  size_t smem = (8 * L.ld + 8) * sizeof(float);
  if (wl) {
    if (L.ld <= 160) AWB_LAUNCH(PK_OUT_LOSS, st, k_out<5, true><<<dim3(S, O), 256, smem, st>>>(q));
    else AWB_LAUNCH(PK_OUT_LOSS, st, k_out<9, true><<<dim3(S, O), 256, smem, st>>>(q));
  } else {
    if (L.ld <= 160) AWB_LAUNCH(PK_OUT_LOSS, st, k_out<5, false><<<dim3(S, O), 256, smem, st>>>(q));
    else AWB_LAUNCH(PK_OUT_LOSS, st, k_out<9, false><<<dim3(S, O), 256, smem, st>>>(q));
  }

  for (int i = L.L; i >= 1; i--) {
    const float* delta = ws.D + (i & 1) * sLayer;
    float* delta_prev = ws.D + ((i - 1) & 1) * sLayer;
    const float* za_prev = ws.ZA + (i - 1) * sLayer;
    const float* W = ws.waug + L.aug_layer + (int64_t)(i - 1) * L.h * L.ld;
    {  // weight gradient: dWaug_i = delta_i^T * ZA_{i-1}
      GemmP p = {};
      p.A = delta; p.sA = sDobj; p.lda = L.ld;
      p.B = za_prev; p.sB = sZAobj; p.ldb = L.ld;
      p.Cout = ws.part + L.aug_layer + (int64_t)(i - 1) * L.h * L.ld; p.sC = L.G; p.ldc = L.ld;
      p.M = L.h; p.N = L.ld; p.K = (int)N;
      p.h = L.h; p.C = L.C; p.k_chunk = chunk; p.sSplit = sSplit;
      AWB_LAUNCH(PK_GEMM_WGRAD, st, k_gemm<2><<<dim3(S, gemm_wgrad_tiles(L), O), 256, 0, st>>>(p));
    }
    {  // data gradient + relu backward
      GemmP p = {};
      p.A = delta; p.sA = sDobj; p.lda = L.ld;
      p.B = W; p.sB = L.G; p.ldb = L.ld;
      p.Cout = delta_prev; p.sC = sDobj; p.ldc = L.ld;
      p.M = N; p.N = L.ld; p.K = L.h;
      p.E0 = za_prev; p.sE0 = sZAobj;
      p.E1 = need_dx ? ws.dX : nullptr; p.sE1 = N * 4;
      p.h = L.h; p.C = L.C;
      AWB_LAUNCH(PK_GEMM_DGRAD, st, k_gemm<1><<<dim3((unsigned)((N + 127) / 128), gemm_col_tiles(L), O), 256, 0, st>>>(p));
    }
  }
  AWB_LAUNCH(PK_IN_BWD, st, k_in_wgrad<<<dim3(S, O), 256, 0, st>>>(ws.D, sDobj, ws.X, ws.part, sSplit, L.G, L.aug_in, N, chunk, L.h, L.ld, 1.f));
  if (need_dx)
    AWB_LAUNCH(PK_IN_BWD, st, k_in_dgrad<<<dim3((unsigned)((N + 7) / 8), O), 256, 0, st>>>(ws.D, sDobj, ws.waug, L.G, L.aug_in, ws.dX, N,
                                                                 L.h, L.ld));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

// Second-order pass of the ICNN's coordinate gradient (DESIGN 3b.1).  The first backward maps (w = dlogits, params) to
// dgrid_n = w_n J_n^T; for a cotangent u on dgrid it returns ydot_n = J_n u_n (to w) and sum_n w_n d(J_n u_n)/d params.
// The relu masks are piecewise constant, so the backprop of the tangent network seeded with w has the deltas of the
// first backward; the weight gradients contract them with the tangent rows ZT instead of the activation rows ZA, and
// every bias gradient is exactly 0.  Reads ZA / X / waug of the training forward, writes ZT, D, dX (as u rows) and part.
int simt_grid_grad_backward(const awb_prior* h, const awb_grid_spec* g, const float* dlogits, const float* d_dgrid,
                            float* ydot, const Workspace& ws, cudaStream_t st) {
  const Layout& L = h->lay;
  const int64_t N = ws.N;
  const int S = n_splits(N);
  const int64_t chunk = split_chunk(N);
  const int64_t sLayer = N * L.ld;
  const int64_t sSplit = L.G;    // one object
  GridDev gu = to_dev(g, L.C, 0);
  gu.mode = AWB_GRID_EXPLICIT; gu.grid = d_dgrid;
  AWB_LAUNCH(PK_TAN_FWD, st, k_tan_input<<<(unsigned)((N + 63) / 64), 256, 0, st>>>(gu, ws.waug, ws.ZA, ws.ZT, ws.dX, N, L.h,
                                                                                 L.C, L.ld, L.aug_in));
  for (int i = 0; i < L.L; i++) {
    GemmP p = {};
    p.A = ws.ZT + i * sLayer; p.lda = L.ld;
    p.B = ws.waug + L.aug_layer + (int64_t)i * L.h * L.ld; p.ldb = L.ld;
    p.Cout = ws.ZT + (i + 1) * sLayer; p.ldc = L.ld;
    p.M = N; p.N = L.h; p.K = L.ld;
    p.E0 = p.A;
    p.Mz = ws.ZA + (i + 1) * sLayer;
    p.h = L.h; p.C = L.C;
    AWB_LAUNCH(PK_TAN_FWD, st, k_gemm<3><<<dim3((unsigned)((N + 127) / 128), gemm_col_tiles(L), 1), 256, 0, st>>>(p));
  }
  TanOutP q = {};
  q.ZA = ws.ZA + L.L * sLayer; q.ZT = ws.ZT + L.L * sLayer;
  q.waug = ws.waug; q.aug_out = L.aug_out;
  q.w = dlogits; q.ydot = ydot;
  q.D = ws.D + (L.L & 1) * sLayer;
  q.part = ws.part; q.sSplit = sSplit;
  q.N = N; q.chunk = chunk; q.h = L.h; q.ld = L.ld;
  const size_t smem = 8 * L.ld * sizeof(float);
  if (L.ld <= 160) AWB_LAUNCH(PK_TAN_OUT, st, k_tan_out<5><<<S, 256, smem, st>>>(q));
  else AWB_LAUNCH(PK_TAN_OUT, st, k_tan_out<9><<<S, 256, smem, st>>>(q));
  for (int i = L.L; i >= 1; i--) {
    const float* delta = ws.D + (i & 1) * sLayer;
    {  // dWaug_i = delta_i^T * ZT_{i-1}
      GemmP p = {};
      p.A = delta; p.lda = L.ld;
      p.B = ws.ZT + (i - 1) * sLayer; p.ldb = L.ld;
      p.Cout = ws.part + L.aug_layer + (int64_t)(i - 1) * L.h * L.ld; p.ldc = L.ld;
      p.M = L.h; p.N = L.ld; p.K = (int)N;
      p.h = L.h; p.C = L.C; p.k_chunk = chunk; p.sSplit = sSplit;
      AWB_LAUNCH(PK_GEMM_WGRAD, st, k_gemm<2><<<dim3(S, gemm_wgrad_tiles(L), 1), 256, 0, st>>>(p));
    }
    {  // delta_{i-1}: the data gradient of the first backward (no coordinate gradient)
      GemmP p = {};
      p.A = delta; p.lda = L.ld;
      p.B = ws.waug + L.aug_layer + (int64_t)(i - 1) * L.h * L.ld; p.ldb = L.ld;
      p.Cout = ws.D + ((i - 1) & 1) * sLayer; p.ldc = L.ld;
      p.M = N; p.N = L.ld; p.K = L.h;
      p.E0 = ws.ZA + (i - 1) * sLayer;
      p.h = L.h; p.C = L.C;
      AWB_LAUNCH(PK_GEMM_DGRAD, st, k_gemm<1><<<dim3((unsigned)((N + 127) / 128), gemm_col_tiles(L), 1), 256, 0, st>>>(p));
    }
  }
  AWB_LAUNCH(PK_IN_BWD, st, k_in_wgrad<<<dim3(S, 1), 256, 0, st>>>(ws.D, 2 * sLayer, ws.dX, ws.part, sSplit, L.G, L.aug_in, N,
                                                                    chunk, L.h, L.ld, 0.f));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

static int n_groups_of(const awb_prior*) { return AWB_MAX_GROUPS; }   // ReduceLROnPlateau reduces every param group (incl. the weight_g group 3)

int simt_reduce_opt(const awb_prior* h, float* params, void* opt_state, const awb_opt_hyper* hy,
                    float* loss_out, const Workspace& ws, int64_t N, cudaStream_t st, int n_partials) {
  const Layout& L = h->lay;
  const int O = h->desc.n_objects;
  OptP a = {};
  a.params = params;
  opt_ptrs(h, opt_state, &a.m, &a.v, &a.scal);
  a.part = ws.part; a.sSplit = (int64_t)O * L.G; a.S = n_partials;
  a.SF = n_splits(N);
  a.PF = L.P_flow + L.n_lin;
  a.fpart = ws.fpart; a.sFSplit = (int64_t)O * a.PF;
  a.lossp = ws.lossp; a.sLoss = O; a.grads = nullptr;
  a.map = h->d_map; a.clamp = h->d_clamp; a.group = h->d_group;
  a.P = L.P; a.off_icnn = L.off_icnn; a.P_icnn = L.P_icnn; a.off_flow = L.off_flow; a.G = L.G;
  a.O = O; a.hy = *hy; a.loss_out = loss_out;
  // augmented-space kernel (programmatic dependent launch, fp16 weight image kept in step): plain ICNN priors, and flow
  // priors whose optimizer owns every group (the flow / linear parameters then ride in extra blocks of the same launch)
  const bool flow_aug = has_flow(h) && hy->active_groups == 0;
  if (h->desc.kind == AWB_KIND_ICNN || flow_aug) {
    OptA b = {};
    b.params = params; b.m = a.m; b.v = a.v; b.scal = a.scal;
    b.part = a.part; b.sSplit = a.sSplit; b.S = a.S; b.lossp = a.lossp;
    b.imap = h->d_imap; b.clamp = h->d_clamp; b.group = h->d_group;
    b.P = L.P; b.off_icnn = L.off_icnn; b.G = L.G; b.aug_out = L.aug_out; b.O = O; b.ld = L.ld;
    b.hy = *hy; b.loss_out = loss_out;
    if (ws.tc && h->d_aug2img) {
      b.img = (uint8_t*)ws.tc; b.img_stride = tc_image_bytes(L.L); b.vec_off = tc_vec_offset_bytes(L.L); b.aug2img = h->d_aug2img;
    }
    unsigned nb = (unsigned)((L.G + 127) / 128);
    if (flow_aug) {
      b.fpart = a.fpart; b.sFSplit = a.sFSplit; b.off_flow = L.off_flow; b.PF = a.PF; b.SF = a.SF; b.nb_aug = (int)nb;
      nb += (unsigned)((a.PF + 127) / 128);
    }
    AWB_LAUNCH(PK_OPT, st, AWB_CUDA(launch_ex(k_reduce_opt_aug, dim3(nb, O), dim3(256), 0, st, true, b, n_groups_of(h))));
  } else {
    AWB_LAUNCH(PK_OPT, st, k_reduce_opt<<<dim3((unsigned)((L.P + 31) / 32), O), 256, 0, st>>>(a, n_groups_of(h), 1));
  }
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int reduce_opt_plain(const awb_prior* h, float* params, void* opt_state, const awb_opt_hyper* hy, float* loss_out,
                     const float* partials, int S, int64_t part_stride, const float* lossp, int64_t loss_stride,
                     cudaStream_t st) {
  const Layout& L = h->lay;
  OptP a = {};
  a.params = params;
  opt_ptrs(h, opt_state, &a.m, &a.v, &a.scal);
  a.part = nullptr; a.sSplit = 0; a.S = 0;
  a.fpart = partials; a.PF = L.P; a.sFSplit = part_stride; a.SF = S;
  a.lossp = lossp; a.sLoss = loss_stride; a.grads = nullptr;
  a.map = nullptr; a.clamp = h->d_clamp; a.group = h->d_group;
  a.P = L.P; a.off_icnn = 0; a.P_icnn = 0; a.off_flow = 0; a.G = 0;
  a.O = 1; a.hy = *hy; a.loss_out = loss_out;
  AWB_LAUNCH(PK_OPT, st, k_reduce_opt<<<dim3((unsigned)((L.P + 31) / 32), 1), 256, 0, st>>>(a, AWB_MAX_GROUPS, 1));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int simt_reduce_grads(const awb_prior* h, float* grads, const Workspace& ws, int64_t N, cudaStream_t st, int n_partials,
                      float* loss_slot) {
  const Layout& L = h->lay;
  const int O = h->desc.n_objects;
  if (loss_slot && O != 1) { set_error("internal: a gradient row is single-object"); return AWB_ERR_INVALID; }
  int64_t PF = L.P_flow + L.n_lin;
  const int64_t n_thr = L.P + (loss_slot ? 1 : 0);
  AWB_LAUNCH(PK_OPT, st, AWB_CUDA(launch_ex(k_reduce_grads, dim3((unsigned)((n_thr + 255) / 256), O), dim3(256), 0, st, true,
      grads, (const float*)ws.part, (int64_t)O * L.G, n_partials, n_splits(N),
      (const float*)ws.fpart, (int64_t)O * PF, (const int32_t*)h->d_map, (int64_t)L.P, (int64_t)L.off_icnn,
      (int64_t)L.P_icnn, (int64_t)L.off_flow, PF, (int64_t)L.G, (const float*)ws.lossp, loss_slot)));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int reduce_grads_plain(const awb_prior* h, float* grads, const float* partials, int S, int64_t part_stride, cudaStream_t st) {
  const int64_t P = h->lay.P;   // no augmented ICNN partials: every entry is read from the plain partials
  AWB_LAUNCH(PK_OPT, st, AWB_CUDA(launch_ex(k_reduce_grads, dim3((unsigned)((P + 255) / 256), 1), dim3(256), 0, st, true,
      grads, (const float*)nullptr, (int64_t)0, 0, S, partials, part_stride, (const int32_t*)nullptr, P, (int64_t)0,
      (int64_t)0, (int64_t)0, P, (int64_t)0, (const float*)nullptr, (float*)nullptr)));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int simt_seed_dX(const awb_prior* h, const float* d_deformed, const Workspace& ws, cudaStream_t st) {
  AWB_LAUNCH(PK_MISC, st, k_seed_dX<<<(unsigned)((ws.N + 255) / 256), 256, 0, st>>>(d_deformed, ws.dX, ws.N, h->lay.C));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int simt_dgrid(const awb_prior* h, const awb_grid_spec* g, float* dgrid, const Workspace& ws, cudaStream_t st) {
  const int64_t N = (int64_t)g->B * g->H * g->W;
  AWB_LAUNCH(PK_MISC, st, k_dgrid<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(ws.dX, dgrid, N, (int64_t)g->H * g->W, h->lay.C));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int optim_step(const awb_prior* h, float* params, const float* grads, void* opt_state,
               const awb_opt_hyper* hy, cudaStream_t st) {
  const Layout& L = h->lay;
  const int O = h->desc.n_objects;
  OptP a = {};
  a.params = params;
  opt_ptrs(h, opt_state, &a.m, &a.v, &a.scal);
  a.grads = grads; a.lossp = nullptr;
  a.map = h->d_map; a.clamp = h->d_clamp; a.group = h->d_group;
  a.P = L.P; a.off_icnn = L.off_icnn; a.P_icnn = L.P_icnn; a.off_flow = L.off_flow; a.G = L.G;
  a.O = O; a.hy = *hy;
  AWB_LAUNCH(PK_OPT, st, k_reduce_opt<<<dim3((unsigned)((L.P + 31) / 32), O), 256, 0, st>>>(a, n_groups_of(h), 0));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

// ReduceLROnPlateau.step(loss) without an optimizer step (one thread per object)
__global__ void k_plateau_step(OptScal* scal, const float* loss, int stride, awb_opt_hyper hy, int n_groups, int O) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= O) return;
  OptScal& s = scal[o];
  const double cur = (double)loss[(int64_t)o * stride];
  if (!isfinite(cur)) { s.nonfinite = 1; return; }
  if (cur < s.best * (1.0 - (double)hy.threshold)) { s.best = cur; s.num_bad = 0; }
  else s.num_bad += 1;
  if (s.num_bad > hy.patience) {
    for (int g = 0; g < n_groups; g++) {
      double nl = s.lr[g] * (double)hy.factor;
      if (nl < (double)hy.min_lr) nl = (double)hy.min_lr;
      if (s.lr[g] - nl > (double)hy.plateau_eps) s.lr[g] = nl;
    }
    s.num_bad = 0;
  }
}

int plateau_step(const awb_prior* h, void* opt_state, const float* loss, int stride, const awb_opt_hyper* hy, cudaStream_t st) {
  float *m, *v;
  OptScal* scal;
  opt_ptrs(h, opt_state, &m, &v, &scal);
  const int O = h->desc.n_objects;
  AWB_LAUNCH(PK_OPT, st, k_plateau_step<<<(O + 31) / 32, 32, 0, st>>>(scal, loss, stride, *hy, n_groups_of(h), O));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int clamp_only(const awb_prior* h, float* params, cudaStream_t st) {
  AWB_LAUNCH(PK_OPT, st, k_clamp<<<dim3((unsigned)((h->lay.P + 255) / 256), h->desc.n_objects), 256, 0, st>>>(params, h->d_clamp, h->lay.P));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int opt_set_lr(const awb_prior* h, void* opt_state, const double* lr, cudaStream_t st) {
  float* m; float* v; OptScal* sc;
  opt_ptrs(h, opt_state, &m, &v, &sc);
  AWB_LAUNCH(PK_MISC, st, k_opt_set_lr<<<1, 64, 0, st>>>(sc, lr[0], lr[1], lr[2], lr[3], h->desc.n_objects));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int opt_state_init(const awb_prior* h, void* opt_state, const double* lr, cudaStream_t st) {
  int64_t n = h->lay.P * h->desc.n_objects;
  float* m; float* v; OptScal* sc;
  opt_ptrs(h, opt_state, &m, &v, &sc);
  AWB_CUDA(cudaMemsetAsync(opt_state, 0, 2 * n * sizeof(float), st));
  AWB_LAUNCH(PK_MISC, st, k_opt_init<<<1, 64, 0, st>>>(sc, lr[0], lr[1], lr[2], lr[3], h->desc.n_objects));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

}  // namespace awb
