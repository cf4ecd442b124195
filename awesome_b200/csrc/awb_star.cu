// Star-shape prior (SURVEY a16): the network ``myNet`` of notebooks/icml_teaser_code/star_shaped/star.ipynb cell 2
//   x <- x + offset;  r = ||x||;  u = x / (0.01 + r);  a = relu(W0 u + b0);
//   b = relu(W1 a + b1 + W1_r r + b1_r);  y = r * (W2 a + b2 + W2_r b + b2_r) - 1
// and the body of its training loop (cell 3): sigmoid + MSE on a sampled point set, backward, Adam, clamp of
// W2_r.weight.  The point sets are small (1000 samples per step in the notebook), so the step is latency bound:
// ONE fused kernel does forward + loss + backward for its slice of the points with one thread per hidden unit,
// W1 and its gradient accumulator resident in shared memory ((h+1)-padded rows: row and column walks are both
// bank-conflict free), cross-thread sums by warp shuffles; per-CTA partials are reduced in a fixed order by the
// shared optimizer kernel (no atomics).
#include <math.h>

#include "awb_internal.cuh"

namespace awb {

struct StarP {
  const float* params; int64_t P; int h;
  const float* x;        // [n][2]
  const float* target;   // [n] (fit)
  int64_t n, chunk;
  LossCoef loss;
  float* logits;         // [n] or null
  float* part;           // [S][P] (fit)
  float* lossp;          // [S]
};

// sum of up to 3 values over the whole block (blockDim.x = 160 = 5 warps); result in every thread
__device__ __forceinline__ void block_sum3(float& a, float& b, float& c, float (*red)[3]) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, off);
    b += __shfl_xor_sync(0xffffffffu, b, off);
    c += __shfl_xor_sync(0xffffffffu, c, off);
  }
  const int w = threadIdx.x >> 5;
  __syncthreads();                       // previous readers of red are done
  if ((threadIdx.x & 31) == 0) { red[w][0] = a; red[w][1] = b; red[w][2] = c; }
  __syncthreads();
  a = b = c = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); i++) { a += red[i][0]; b += red[i][1]; c += red[i][2]; }   // fixed order
}

template <bool FIT>
__global__ void __launch_bounds__(160) k_star(StarP p) {
  extern __shared__ float sm[];
  const int h = p.h, ld = h + 1;
  float* sW1 = sm;                       // [h][h+1]
  float* sG = sm + h * ld;               // [h][h+1] gradient accumulator (FIT)
  float* sa = sG + (FIT ? h * ld : 0);   // [h]
  float* sdb = sa + h;                   // [h]
  __shared__ float red[8][3];
  const int j = threadIdx.x;
  const bool act = j < h;
  const float* par = p.params;
  const int o_W0 = 2, o_b0 = 2 + 2 * h, o_W1 = 2 + 3 * h, o_b1 = o_W1 + h * h, o_W2 = o_b1 + h, o_b2 = o_W2 + h,
            o_W1r = o_b2 + 1, o_b1r = o_W1r + h, o_W2r = o_b1r + h, o_b2r = o_W2r + h;
  for (int i = threadIdx.x; i < h * h; i += blockDim.x) { sW1[(i / h) * ld + (i % h)] = par[o_W1 + i]; }
  if (FIT) for (int i = threadIdx.x; i < h * ld; i += blockDim.x) sG[i] = 0.f;
  const float off0 = par[0], off1 = par[1];
  float w0x = 0.f, w0y = 0.f, b0 = 0.f, w1r = 0.f, bb1 = 0.f, w2 = 0.f, w2r = 0.f;
  if (act) {
    w0x = par[o_W0 + 2 * j]; w0y = par[o_W0 + 2 * j + 1]; b0 = par[o_b0 + j];
    w1r = par[o_W1r + j]; bb1 = par[o_b1 + j] + par[o_b1r + j];
    w2 = par[o_W2 + j]; w2r = par[o_W2r + j];
  }
  const float bias2 = par[o_b2] + par[o_b2r];
  float g_w0x = 0.f, g_w0y = 0.f, g_b0 = 0.f, g_w1r = 0.f, g_b1 = 0.f, g_w2 = 0.f, g_w2r = 0.f;
  float g_b2 = 0.f, g_ox = 0.f, g_oy = 0.f, lacc = 0.f;
  __syncthreads();
  const int64_t r0 = (int64_t)blockIdx.x * p.chunk, r1 = r0 + p.chunk < p.n ? r0 + p.chunk : p.n;
  for (int64_t pt = r0; pt < r1; pt++) {
    const float px = p.x[2 * pt] + off0, py = p.x[2 * pt + 1] + off1;
    const float r = sqrtf(px * px + py * py), q = 0.01f + r;
    const float ux = px / q, uy = py / q;
    const float apre = act ? fmaf(w0x, ux, fmaf(w0y, uy, b0)) : 0.f;
    const float a = fmaxf(apre, 0.f);
    if (act) sa[j] = a;
    __syncthreads();
    float bpre = 0.f;
    if (act) {
      bpre = fmaf(w1r, r, bb1);
      const float* wr = sW1 + j * ld;
#pragma unroll 5
      for (int k = 0; k < h; k++) bpre = fmaf(wr[k], sa[k], bpre);
    }
    const float b = fmaxf(bpre, 0.f);
    float s = act ? fmaf(w2, a, w2r * b) : 0.f, z1 = 0.f, z2 = 0.f;
    block_sum3(s, z1, z2, red);
    s += bias2;
    const float y = fmaf(r, s, -1.f);
    if (p.logits && j == 0) p.logits[pt] = y;
    if (!FIT) continue;
    const float t = p.target[pt];
    const bool fg = p.loss.cls_rule == AWB_CLS_UNARY_LT_HALF ? (t < 0.5f) : (t != 1.0f);
    const float coef = fg ? p.loss.coef_fg : p.loss.coef_bg;
    const float sg = 1.f / (1.f + expf(-y));
    float l, dl;
    if (p.loss.kind == AWB_LOSS_SE_SIGMOID) { float d = t - sg; l = d * d; dl = -2.f * d * sg * (1.f - sg); }
    else { l = fmaxf(y, 0.f) - y * t + log1pf(expf(-fabsf(y))); dl = sg - t; }
    const float dy = coef * dl, dyr = dy * r;
    float db = 0.f;
    if (act) {
      g_w2 = fmaf(dyr, a, g_w2); g_w2r = fmaf(dyr, b, g_w2r);
      db = bpre > 0.f ? dyr * w2r : 0.f;
      g_b1 += db; g_w1r = fmaf(db, r, g_w1r);
      sdb[j] = db;
      float* gr = sG + j * ld;
#pragma unroll 5
      for (int k = 0; k < h; k++) gr[k] = fmaf(db, sa[k], gr[k]);
    }
    __syncthreads();
    float dapre = 0.f;
    if (act) {
      float da = dyr * w2;
#pragma unroll 5
      for (int i = 0; i < h; i++) da = fmaf(sdb[i], sW1[i * ld + j], da);
      dapre = apre > 0.f ? da : 0.f;
      g_w0x = fmaf(dapre, ux, g_w0x); g_w0y = fmaf(dapre, uy, g_w0y); g_b0 += dapre;
    }
    float dux = dapre * w0x, duy = dapre * w0y, drb = db * w1r;
    block_sum3(dux, duy, drb, red);
    if (j == 0) {
      lacc = fmaf(coef, l, lacc);
      g_b2 += dyr;
      if (r > 0.f) {
        const float dr = fmaf(dy, s, drb) - (dux * px + duy * py) / (q * q);
        g_ox += dux / q + dr * (px / r);
        g_oy += duy / q + dr * (py / r);
      }
    }
    __syncthreads();     // sa / sdb are rewritten by the next point
  }
  if (!FIT) return;
  __syncthreads();
  float* out = p.part + (int64_t)blockIdx.x * p.P;
  if (act) {
    out[o_W0 + 2 * j] = g_w0x; out[o_W0 + 2 * j + 1] = g_w0y; out[o_b0 + j] = g_b0;
    out[o_b1 + j] = g_b1; out[o_b1r + j] = g_b1; out[o_W1r + j] = g_w1r;
    out[o_W2 + j] = g_w2; out[o_W2r + j] = g_w2r;
  }
  if (j == 0) { out[0] = g_ox; out[1] = g_oy; out[o_b2] = g_b2; out[o_b2r] = g_b2; p.lossp[blockIdx.x] = lacc; }
  for (int i = threadIdx.x; i < h * h; i += blockDim.x) out[o_W1 + i] = sG[(i / h) * ld + (i % h)];
}

int star_n_ctas(int64_t n) {
  int64_t c = (n + 3) / 4;
  return (int)(c < 1 ? 1 : (c > kMaxSplits ? kMaxSplits : c));
}

int star_run(const awb_prior* h, const float* params, const float* x, const float* target, int64_t n,
             const awb_loss_spec* loss, float* logits, float* part, float* lossp, bool fit, int* n_ctas, cudaStream_t st) {
  const int hh = h->lay.h;
  if (hh > 160) { set_error("star prior supports n_hidden <= 160, got %d", hh); return AWB_ERR_UNSUPPORTED; }
  StarP p = {};
  p.params = params; p.P = h->lay.P; p.h = hh; p.x = x; p.target = target; p.n = n;
  const int S = fit ? star_n_ctas(n) : (int)((n + 15) / 16 < 1184 ? (n + 15) / 16 : 1184);
  p.chunk = (n + S - 1) / S;
  if (loss) p.loss = loss_coef(*loss);
  p.logits = logits; p.part = part; p.lossp = lossp;
  const size_t smem = sizeof(float) * ((size_t)(fit ? 2 : 1) * hh * (hh + 1) + 2 * hh);
  if (fit) {
    AWB_CUDA(cudaFuncSetAttribute(k_star<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    AWB_LAUNCH(PK_MISC, st, k_star<true><<<S, 160, smem, st>>>(p));
  } else {
    AWB_CUDA(cudaFuncSetAttribute(k_star<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    AWB_LAUNCH(PK_MISC, st, k_star<false><<<S, 160, smem, st>>>(p));
  }
  AWB_CUDA(cudaGetLastError());
  if (n_ctas) *n_ctas = S;
  return AWB_OK;
}

// ---- backward for an upstream gradient per point (awb_star_backward): the autograd path of StarShapedNet.
// k_star walks its points one at a time with block barriers in between, which is fine for the notebook's 1000 samples
// but serial at a full frame (307 200 points = ~2000 points per CTA).  k_star_bwd works on a tile of kStarT points per
// iteration instead.  Each warp owns kStarTM points of the tile and each lane the hidden units l + 32 u (u < NU), so
//   bpre = W1 a + W1_r r + b1 + b1_r   and   da = W1^T db + dyr w2
// are register-blocked [kStarTM x NU] products over W1 in shared memory, and the tile's a and db (shared memory, [T][HP])
// feed dW1 += db^T a once per tile, a [HP x T] x [T x HP] contraction whose accumulator stays in registers for the whole
// CTA (thread (jt, kt) owns dW1[jt + 16 a][kt + 16 b]).  Every product is fp32 FMA in k_star's order of operations; the
// sums over points run in point order within the CTA and per-CTA partials are reduced in CTA order (no atomics).
constexpr int kStarT = 64;                       // points per tile
constexpr int kStarWarps = 8;                    // 256 threads
constexpr int kStarTM = kStarT / kStarWarps;     // points per warp in the two W1 products
enum { SP_W0X = 0, SP_W0Y, SP_B0, SP_W1R, SP_B1, SP_W2, SP_W2R, SP_N };           // per-unit parameters (sPar rows)
enum { SG_W0X = 0, SG_W0Y, SG_B0, SG_B1, SG_W1R, SG_W2, SG_W2R, SG_N };           // per-unit gradient sums (sAcc rows)
enum { PT_PX = 0, PT_PY, PT_R, PT_Q, PT_UX, PT_UY, PT_DY, PT_DYR, PT_N };         // per-point values (sPt rows)

struct StarBwdP {
  const float* params; int64_t P; int h;
  const float* x;        // [n][2]
  const float* dy;       // [n]
  int64_t n, chunk;      // chunk: points per CTA, a multiple of kStarT
  float* part;           // [S][P]
  float* dx;             // [n][2] or null
};

template <int NU>
constexpr size_t star_bwd_smem() {
  return sizeof(float) * ((size_t)32 * NU * (32 * NU + 4) + 2 * kStarT * 32 * NU + (size_t)(kStarWarps * SG_N + SP_N) * 32 * NU +
                          PT_N * kStarT);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

// The fused fit step on whole frames (awb_prior_fit_step on a star handle): the points are the pixel rows of an explicit
// planar [B,2,H,W] grid and dy comes from the loss on the target, per point, inside the tile.  WL: the loss carries a
// weight map and / or an ignore label (the plain instantiation reads neither).
struct StarFitX {
  GridDev g;             // explicit grid, C = 2
  const float* target;   // [N]
  LossCoef loss;
  LossPix pix;
  float* lossp;          // [S] loss partial per CTA
};

template <bool>
using StarFitArg = StarFitX;
__device__ __forceinline__ StarFitX star_fit_arg() { return StarFitX{}; }
__device__ __forceinline__ StarFitX star_fit_arg(const StarFitX& f) { return f; }

// k_star_bwd<NU> (no fit argument): the backward of awb_star_backward, x [n][2] and dy given.  k_star_bwd<NU, WL> (one
// StarFitX): the fused fit step, the points are grid rows and dy comes from the loss.  The fit mode splits the b / db loop
// in two: pass 1 sums s over the lane's units, the lane that owns the point turns y = r (s + b2 + b2_r) - 1 into its loss
// term and dy, and pass 2 is the backward's loop without the s sum.  The mode is a template parameter pack so that the
// backward's instantiation is the kernel it always was.
template <int NU, bool... WLs>
__global__ void __launch_bounds__(kStarWarps * 32, 1) k_star_bwd(StarBwdP p, StarFitArg<WLs>... fa) {
  static_assert(sizeof...(WLs) <= 1, "one fit argument at most");
  constexpr bool FIT = sizeof...(WLs) == 1, WL = (false || ... || WLs);
  const StarFitX f = star_fit_arg(fa...);
  constexpr int HP = 32 * NU, LDW = HP + 4, T = kStarT, TM = kStarTM;
  extern __shared__ __align__(16) float sm[];
  float* sW1 = sm;                          // [HP][LDW] W1, zero outside [h][h]
  float* sA = sW1 + HP * LDW;               // [T][HP] a of the tile's points (0 for units >= h)
  float* sDB = sA + T * HP;                 // [T][HP] db
  float* sAcc = sDB + T * HP;               // [warp][SG_N][HP] per-unit gradient sums over each warp's points
  float* sPar = sAcc + kStarWarps * SG_N * HP;   // [SP_N][HP], zero for units >= h
  float* sPt = sPar + SP_N * HP;            // [PT_N][T]
  __shared__ float red[kStarWarps][FIT ? 4 : 3];
  const int tid = threadIdx.x, w = tid >> 5, l = tid & 31, h = p.h;
  const float* par = p.params;
  const int o_W0 = 2, o_b0 = 2 + 2 * h, o_W1 = 2 + 3 * h, o_b1 = o_W1 + h * h, o_W2 = o_b1 + h, o_b2 = o_W2 + h,
            o_W1r = o_b2 + 1, o_b1r = o_W1r + h, o_W2r = o_b1r + h, o_b2r = o_W2r + h;
  for (int i = tid; i < HP * LDW; i += blockDim.x) {
    const int j = i / LDW, k = i - j * LDW;
    sW1[i] = (j < h && k < h) ? par[o_W1 + j * h + k] : 0.f;
  }
  for (int i = tid; i < kStarWarps * SG_N * HP; i += blockDim.x) sAcc[i] = 0.f;
  for (int j = tid; j < HP; j += blockDim.x) {
    const bool in = j < h;
    sPar[SP_W0X * HP + j] = in ? par[o_W0 + 2 * j] : 0.f;
    sPar[SP_W0Y * HP + j] = in ? par[o_W0 + 2 * j + 1] : 0.f;
    sPar[SP_B0 * HP + j] = in ? par[o_b0 + j] : 0.f;
    sPar[SP_W1R * HP + j] = in ? par[o_W1r + j] : 0.f;
    sPar[SP_B1 * HP + j] = in ? par[o_b1 + j] + par[o_b1r + j] : 0.f;
    sPar[SP_W2 * HP + j] = in ? par[o_W2 + j] : 0.f;
    sPar[SP_W2R * HP + j] = in ? par[o_W2r + j] : 0.f;
  }
  const float off0 = par[0], off1 = par[1], bias2 = par[o_b2] + par[o_b2r];
  const int Kp = (h + 3) & ~3;              // W1 products run over round_up(h, 4): the padding adds exact zeros
  const int jt = tid >> 4, kt = tid & 15;
  float dW[2 * NU][2 * NU];
#pragma unroll
  for (int a = 0; a < 2 * NU; a++)
#pragma unroll
    for (int b = 0; b < 2 * NU; b++) dW[a][b] = 0.f;
  float g_ox = 0.f, g_oy = 0.f, g_b2 = 0.f;   // lanes < TM: sums over the points they finish
  float lacc = 0.f;                            // FIT: the warp's loss, its points in point order (every lane holds it)
  __syncthreads();
  const int64_t c0 = (int64_t)blockIdx.x * p.chunk, c1 = c0 + p.chunk < p.n ? c0 + p.chunk : p.n;
  for (int64_t t0 = c0; t0 < c1; t0 += T) {
    // remainder tile: only the last tile of the last CTA has nv < T (n % kStarT != 0); its padding points sit at r = 0
    // with dy = 0 and add exact zeros to every sum
    const int nv = (int)(c1 - t0 < T ? c1 - t0 : T);
    if (tid < T) {
      float px = 0.f, py = 0.f, dy = 0.f;
      if (tid < nv) {
        const int64_t n = t0 + tid;
        if (FIT) {
          px = coord(f.g, n, 0) + off0; py = coord(f.g, n, 1) + off1;
        } else {
          px = p.x[2 * n] + off0; py = p.x[2 * n + 1] + off1; dy = p.dy[n];
        }
      }
      const float r = sqrtf(px * px + py * py), q = 0.01f + r;
      sPt[PT_PX * T + tid] = px; sPt[PT_PY * T + tid] = py; sPt[PT_R * T + tid] = r; sPt[PT_Q * T + tid] = q;
      sPt[PT_UX * T + tid] = px / q; sPt[PT_UY * T + tid] = py / q;
      if (!FIT) { sPt[PT_DY * T + tid] = dy; sPt[PT_DYR * T + tid] = dy * r; }   // FIT: written by the loss lane below
    }
    // FIT: the lane that will finish point w * TM + l fetches its target (and weight) now; the W1 product hides the load
    float tg = 0.f, wt = 1.f;
    if (FIT && l < TM && w * TM + l < nv) {
      const int64_t n = t0 + w * TM + l;
      tg = f.target[n];
      if (WL && f.pix.weight) wt = f.pix.weight[n];
    }
    __syncthreads();
    // a = relu(W0 u + b0) of the warp's points
#pragma unroll
    for (int i = 0; i < TM; i++) {
      const int t = w * TM + i;
      const float ux = sPt[PT_UX * T + t], uy = sPt[PT_UY * T + t];
#pragma unroll
      for (int u = 0; u < NU; u++) {
        const int j = l + 32 * u;
        const float apre = fmaf(sPar[SP_W0X * HP + j], ux, fmaf(sPar[SP_W0Y * HP + j], uy, sPar[SP_B0 * HP + j]));
        sA[t * HP + j] = fmaxf(apre, 0.f);
      }
    }
    __syncwarp();
    // bpre = W1_r r + b1 + b1_r + W1 a
    float acc[TM][NU];
#pragma unroll
    for (int i = 0; i < TM; i++)
#pragma unroll
      for (int u = 0; u < NU; u++)
        acc[i][u] = fmaf(sPar[SP_W1R * HP + l + 32 * u], sPt[PT_R * T + w * TM + i], sPar[SP_B1 * HP + l + 32 * u]);
    for (int k = 0; k < Kp; k += 4) {
      float4 wv[NU];
#pragma unroll
      for (int u = 0; u < NU; u++) wv[u] = *reinterpret_cast<const float4*>(sW1 + (l + 32 * u) * LDW + k);
#pragma unroll
      for (int i = 0; i < TM; i++) {
        const float4 a4 = *reinterpret_cast<const float4*>(sA + (w * TM + i) * HP + k);
#pragma unroll
        for (int u = 0; u < NU; u++) {
          acc[i][u] = fmaf(wv[u].x, a4.x, acc[i][u]); acc[i][u] = fmaf(wv[u].y, a4.y, acc[i][u]);
          acc[i][u] = fmaf(wv[u].z, a4.z, acc[i][u]); acc[i][u] = fmaf(wv[u].w, a4.w, acc[i][u]);
        }
      }
    }
    float s_me = 0.f, drb_me = 0.f;   // lane i < TM keeps point w * TM + i
    if (FIT) {
      // pass 1: s = sum_j w2_j a_j + w2r_j b_j per point, then the loss of the lane's point and its dy
      float s[TM];
#pragma unroll
      for (int i = 0; i < TM; i++) s[i] = 0.f;
#pragma unroll
      for (int u = 0; u < NU; u++) {
        const int j = l + 32 * u;
        const float w2 = sPar[SP_W2 * HP + j], w2r = sPar[SP_W2R * HP + j];
#pragma unroll
        for (int i = 0; i < TM; i++) s[i] += fmaf(w2, sA[(w * TM + i) * HP + j], w2r * fmaxf(acc[i][u], 0.f));
      }
#pragma unroll
      for (int i = 0; i < TM; i++) {
        const float si = warp_sum(s[i]);
        if (l == i) s_me = si;
      }
      // k_star's loss: SE on the sigmoid or BCE with logits, coef by cls_rule (times the weight); padding points and
      // (WL) ignored pixels are selected out, so their dy and loss term are exactly 0 whatever their inputs
      float lterm = 0.f;
      if (l < TM) {
        const int t = w * TM + l;
        const float r = sPt[PT_R * T + t];
        const float y = fmaf(r, s_me + bias2, -1.f);
        const bool fg = f.loss.cls_rule == AWB_CLS_UNARY_LT_HALF ? (tg < 0.5f) : (tg != 1.0f);
        float coef = fg ? f.loss.coef_fg : f.loss.coef_bg;
        if (WL) coef *= wt;
        const float sg = 1.f / (1.f + expf(-y));
        float lv, dl;
        if (f.loss.kind == AWB_LOSS_SE_SIGMOID) { const float d = tg - sg; lv = d * d; dl = -2.f * d * sg * (1.f - sg); }
        else { lv = fmaxf(y, 0.f) - y * tg + log1pf(expf(-fabsf(y))); dl = sg - tg; }
        const bool keep = t < nv && (!WL || loss_keep(f.pix, tg));
        const float dy = keep ? coef * dl : 0.f;
        lterm = keep ? coef * lv : 0.f;
        sPt[PT_DY * T + t] = dy; sPt[PT_DYR * T + t] = dy * r;
      }
#pragma unroll
      for (int i = 0; i < TM; i++) lacc += __shfl_sync(0xffffffffu, lterm, i);
      __syncwarp();
    }
    // b, db; (BWD: s and) drb = sum_j db_j w1r_j per point; the per-unit sums of dyr a, dyr b, db, db r
    float s[TM], drb[TM];
#pragma unroll
    for (int i = 0; i < TM; i++) { s[i] = 0.f; drb[i] = 0.f; }
#pragma unroll
    for (int u = 0; u < NU; u++) {
      const int j = l + 32 * u;
      const float w2 = sPar[SP_W2 * HP + j], w2r = sPar[SP_W2R * HP + j], w1r = sPar[SP_W1R * HP + j];
      float* ga = sAcc + w * SG_N * HP + j;
      float g_w2 = ga[SG_W2 * HP], g_w2r = ga[SG_W2R * HP], g_b1 = ga[SG_B1 * HP], g_w1r = ga[SG_W1R * HP];
#pragma unroll
      for (int i = 0; i < TM; i++) {
        const int t = w * TM + i;
        const float a = sA[t * HP + j], b = fmaxf(acc[i][u], 0.f);
        const float dyr = sPt[PT_DYR * T + t], r = sPt[PT_R * T + t];
        if (!FIT) s[i] += fmaf(w2, a, w2r * b);
        const float db = acc[i][u] > 0.f ? dyr * w2r : 0.f;
        sDB[t * HP + j] = db;
        drb[i] = fmaf(db, w1r, drb[i]);
        g_w2 = fmaf(dyr, a, g_w2); g_w2r = fmaf(dyr, b, g_w2r);
        g_b1 += db; g_w1r = fmaf(db, r, g_w1r);
      }
      ga[SG_W2 * HP] = g_w2; ga[SG_W2R * HP] = g_w2r; ga[SG_B1 * HP] = g_b1; ga[SG_W1R * HP] = g_w1r;
    }
#pragma unroll
    for (int i = 0; i < TM; i++) {
      if (FIT) {
        const float di = warp_sum(drb[i]);
        if (l == i) drb_me = di;
      } else {
        const float si = warp_sum(s[i]), di = warp_sum(drb[i]);
        if (l == i) { s_me = si; drb_me = di; }
      }
    }
    __syncwarp();
    // da = dyr w2 + W1^T db; dapre; the per-unit sums of dapre ux, dapre uy, dapre; du = W0^T dapre per point
#pragma unroll
    for (int i = 0; i < TM; i++)
#pragma unroll
      for (int u = 0; u < NU; u++) acc[i][u] = sPt[PT_DYR * T + w * TM + i] * sPar[SP_W2 * HP + l + 32 * u];
    for (int j = 0; j < Kp; j += 4) {
      float wv[4][NU];
#pragma unroll
      for (int c = 0; c < 4; c++)
#pragma unroll
        for (int u = 0; u < NU; u++) wv[c][u] = sW1[(j + c) * LDW + l + 32 * u];
#pragma unroll
      for (int i = 0; i < TM; i++) {
        const float4 d4 = *reinterpret_cast<const float4*>(sDB + (w * TM + i) * HP + j);
#pragma unroll
        for (int u = 0; u < NU; u++) {
          acc[i][u] = fmaf(d4.x, wv[0][u], acc[i][u]); acc[i][u] = fmaf(d4.y, wv[1][u], acc[i][u]);
          acc[i][u] = fmaf(d4.z, wv[2][u], acc[i][u]); acc[i][u] = fmaf(d4.w, wv[3][u], acc[i][u]);
        }
      }
    }
    float dux[TM], duy[TM];
#pragma unroll
    for (int i = 0; i < TM; i++) { dux[i] = 0.f; duy[i] = 0.f; }
#pragma unroll
    for (int u = 0; u < NU; u++) {
      const int k = l + 32 * u;
      const float w0x = sPar[SP_W0X * HP + k], w0y = sPar[SP_W0Y * HP + k];
      float* ga = sAcc + w * SG_N * HP + k;
      float g_w0x = ga[SG_W0X * HP], g_w0y = ga[SG_W0Y * HP], g_b0 = ga[SG_B0 * HP];
#pragma unroll
      for (int i = 0; i < TM; i++) {
        const int t = w * TM + i;
        const float dapre = sA[t * HP + k] > 0.f ? acc[i][u] : 0.f;   // a > 0 exactly where its pre-activation is
        g_w0x = fmaf(dapre, sPt[PT_UX * T + t], g_w0x); g_w0y = fmaf(dapre, sPt[PT_UY * T + t], g_w0y); g_b0 += dapre;
        dux[i] = fmaf(dapre, w0x, dux[i]); duy[i] = fmaf(dapre, w0y, duy[i]);
      }
      ga[SG_W0X * HP] = g_w0x; ga[SG_W0Y * HP] = g_w0y; ga[SG_B0 * HP] = g_b0;
    }
    float dux_me = 0.f, duy_me = 0.f;
#pragma unroll
    for (int i = 0; i < TM; i++) {
      const float xi = warp_sum(dux[i]), yi = warp_sum(duy[i]);
      if (l == i) { dux_me = xi; duy_me = yi; }
    }
    // the point gradient, written once by the lane that finishes the point; the offset's gradient is its sum
    if (l < TM && w * TM + l < nv) {
      const int t = w * TM + l;
      const float px = sPt[PT_PX * T + t], py = sPt[PT_PY * T + t], r = sPt[PT_R * T + t], q = sPt[PT_Q * T + t];
      const float dy = sPt[PT_DY * T + t];
      g_b2 += sPt[PT_DYR * T + t];
      // r = 0 (the point at -offset): no contribution through r, as in k_star; the u path (du/dx = I / 0.01) is kept
      float gx = dux_me / q, gy = duy_me / q;
      if (r > 0.f) {
        const float dr = fmaf(dy, s_me + bias2, drb_me) - (dux_me * px + duy_me * py) / (q * q);
        gx = dux_me / q + dr * (px / r);
        gy = duy_me / q + dr * (py / r);
      }
      g_ox += gx; g_oy += gy;
      if (!FIT && p.dx) { const int64_t n = t0 + t; p.dx[2 * n] = gx; p.dx[2 * n + 1] = gy; }
    }
    __syncthreads();
    // dW1 += db^T a over the tile's points, in point order
    for (int t = 0; t < nv; t++) {
      float dbv[2 * NU], av[2 * NU];
#pragma unroll
      for (int a = 0; a < 2 * NU; a++) { dbv[a] = sDB[t * HP + jt + 16 * a]; av[a] = sA[t * HP + kt + 16 * a]; }
#pragma unroll
      for (int a = 0; a < 2 * NU; a++)
#pragma unroll
        for (int b = 0; b < 2 * NU; b++) dW[a][b] = fmaf(dbv[a], av[b], dW[a][b]);
    }
    __syncthreads();     // the next tile rewrites sPt, sA and sDB
  }
  // this CTA's partial, state_dict order; every sum over warps or lanes in a fixed order
  float* out = p.part + (int64_t)blockIdx.x * p.P;
  for (int j = tid; j < h; j += blockDim.x) {
    float g[SG_N];
#pragma unroll
    for (int q = 0; q < SG_N; q++) {
      g[q] = 0.f;
      for (int v = 0; v < kStarWarps; v++) g[q] += sAcc[(v * SG_N + q) * HP + j];
    }
    out[o_W0 + 2 * j] = g[SG_W0X]; out[o_W0 + 2 * j + 1] = g[SG_W0Y]; out[o_b0 + j] = g[SG_B0];
    out[o_b1 + j] = g[SG_B1]; out[o_b1r + j] = g[SG_B1]; out[o_W1r + j] = g[SG_W1R];
    out[o_W2 + j] = g[SG_W2]; out[o_W2r + j] = g[SG_W2R];
  }
#pragma unroll
  for (int a = 0; a < 2 * NU; a++)
#pragma unroll
    for (int b = 0; b < 2 * NU; b++) {
      const int j = jt + 16 * a, k = kt + 16 * b;
      if (j < h && k < h) out[o_W1 + j * h + k] = dW[a][b];
    }
  g_ox = warp_sum(g_ox); g_oy = warp_sum(g_oy); g_b2 = warp_sum(g_b2);
  if (l == 0) {
    red[w][0] = g_ox; red[w][1] = g_oy; red[w][2] = g_b2;
    if (FIT) red[w][FIT ? 3 : 0] = lacc;
  }
  __syncthreads();
  if (tid == 0) {
    float ox = 0.f, oy = 0.f, b2 = 0.f, ls = 0.f;
    for (int v = 0; v < kStarWarps; v++) {
      ox += red[v][0]; oy += red[v][1]; b2 += red[v][2];
      if (FIT) ls += red[v][FIT ? 3 : 0];
    }
    out[0] = ox; out[1] = oy; out[o_b2] = b2; out[o_b2r] = b2;
    if (FIT) f.lossp[blockIdx.x] = ls;
  }
}


// Launch geometry of k_star_bwd.  Size-dependent branches (tests/test_gpu_star_autograd.py covers both sides of each):
//  - tiles per CTA: ceil(n / kStarT) tiles are dealt to at most kMaxSplits CTAs in runs of ceil(tiles / kMaxSplits):
//    one tile per CTA while n <= kMaxSplits * kStarT = 9472, several above;
//  - CTA count S = ceil(tiles / tiles per CTA) (<= kMaxSplits; no CTA is empty);
//  - remainder tile: n % kStarT != 0 leaves the last tile of the last CTA partial.
int star_bwd_ctas(int64_t n, int64_t* chunk) {
  const int64_t tiles = (n + kStarT - 1) / kStarT, per = (tiles + kMaxSplits - 1) / kMaxSplits;
  if (chunk) *chunk = per * kStarT;
  return (int)((tiles + per - 1) / per);
}

template <int NU>
static int star_bwd_launch(const StarBwdP& p, int S, cudaStream_t st) {
  constexpr size_t smem = star_bwd_smem<NU>();
  static_assert(smem <= 227 * 1024, "k_star_bwd shared memory");
  AWB_CUDA(cudaFuncSetAttribute(k_star_bwd<NU>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  AWB_LAUNCH(PK_STAR_BWD, st, k_star_bwd<NU><<<S, kStarWarps * 32, smem, st>>>(p));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int star_backward(const awb_prior* h, const float* params, const float* x, const float* dy, int64_t n, float* grads,
                  float* dx, float* part, cudaStream_t st) {
  const int hh = h->lay.h;
  if (hh > 160) { set_error("star prior supports n_hidden <= 160, got %d", hh); return AWB_ERR_UNSUPPORTED; }
  StarBwdP p = {};
  p.params = params; p.P = h->lay.P; p.h = hh; p.x = x; p.dy = dy; p.n = n; p.part = part; p.dx = dx;
  const int S = star_bwd_ctas(n, &p.chunk);
  int rc;
  switch ((hh + 31) / 32) {
    case 1: rc = star_bwd_launch<1>(p, S, st); break;
    case 2: rc = star_bwd_launch<2>(p, S, st); break;
    case 3: rc = star_bwd_launch<3>(p, S, st); break;
    case 4: rc = star_bwd_launch<4>(p, S, st); break;
    default: rc = star_bwd_launch<5>(p, S, st); break;
  }
  if (rc) return rc;
  return reduce_grads_plain(h, grads, part, S, h->lay.P, st);
}

template <int NU, bool WL>
static int star_fit_launch(const StarBwdP& p, const StarFitX& f, int S, cudaStream_t st) {
  constexpr size_t smem = star_bwd_smem<NU>();
  AWB_CUDA(cudaFuncSetAttribute(k_star_bwd<NU, WL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  AWB_LAUNCH(PK_STAR_FIT, st, k_star_bwd<NU, WL><<<S, kStarWarps * 32, smem, st>>>(p, f));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

template <bool WL>
static int star_fit_dispatch(int hh, const StarBwdP& p, const StarFitX& f, int S, cudaStream_t st) {
  switch ((hh + 31) / 32) {
    case 1: return star_fit_launch<1, WL>(p, f, S, st);
    case 2: return star_fit_launch<2, WL>(p, f, S, st);
    case 3: return star_fit_launch<3, WL>(p, f, S, st);
    case 4: return star_fit_launch<4, WL>(p, f, S, st);
    default: return star_fit_launch<5, WL>(p, f, S, st);
  }
}

int star_fit(const awb_prior* h, const float* params, const awb_grid_spec* g, const float* target,
             const awb_loss_spec& loss, const Workspace& ws, int* n_ctas, cudaStream_t st) {
  const int hh = h->lay.h;
  if (hh > 160) { set_error("star prior supports n_hidden <= 160, got %d", hh); return AWB_ERR_UNSUPPORTED; }
  StarBwdP p = {};
  p.params = params; p.P = h->lay.P; p.h = hh; p.n = ws.N; p.part = ws.part;
  const int S = star_bwd_ctas(ws.N, &p.chunk);
  StarFitX f = {};
  f.g.mode = g->mode; f.g.B = g->B; f.g.H = g->H; f.g.W = g->W; f.g.C = 2; f.g.grid = g->grid; f.g.row0 = 0;
  f.target = target; f.loss = loss_coef(loss); f.pix = loss_pix(loss); f.lossp = ws.lossp;
  const int rc = loss_is_weighted(loss) ? star_fit_dispatch<true>(hh, p, f, S, st) : star_fit_dispatch<false>(hh, p, f, S, st);
  if (rc) return rc;
  *n_ctas = S;
  return AWB_OK;
}

}  // namespace awb
