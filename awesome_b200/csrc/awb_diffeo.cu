// Coupling flow of the older diffeomorphism prior (SURVEY a6): ConvexDiffeomorphismNet =
//   nn.Linear(C, C) on the coordinates -> NormalizingFlow1D -> ConvexNextNet
// (awesome/model/convex_diffeomorphism_net.py:130-178; awesome/model/diffeomorphism_net.py:83-104,208-300).
// NormalizingFlow1D: num_coupling alternating two-variable couplings
//   i even:  x2 <- exp(c_i * S_i(x1)) * x2 + T_i(x1)        i odd:  x1 <- exp(c_i * S_i(x2)) * x1 + T_i(x2)
// with S_i, T_i = SimpleBackbone: tanh(WN(w,1)( relu( WN(1,w)(x) ) )), WN = weight_norm(Linear, dim=None)
// (W = g * v / ||v||_F, awesome/model/real_nvp/resnet_1d.py:39-63) and the scalar
// c_i = WNScale() = weight_norm(Linear(1,1))(weight_i)  (dim=0: g * v/|v| * weight + bias).
//
// forward : one thread per pixel, effective (de-normalised) weights staged in shared memory; writes the deformed
//           coordinates X[n] = (x1, x2, 0, 1) for the ICNN and the input pair of every coupling for the backward.
// backward: one warp per pixel, lane k owns hidden units k, k+32, k+64 of every backbone: the hidden-unit
//           gradients accumulate in lane-private registers (no atomics, no shared-memory traffic per pixel),
//           the scalar outputs use warp shuffles.  Per-CTA sums are reduced over the warps in a fixed order, pushed
//           through the weight-norm Jacobian (linear, so it commutes with the cross-CTA sum) and written as
//           state_dict-ordered partials for the shared optimizer kernel.
#include <math.h>

#include "awb_internal.cuh"

namespace awb {

namespace {
constexpr int kMaxNC = 8;      // couplings
}

struct DiffP {
  GridDev g;
  const float* params; int64_t P, off_flow, PF;
  int nc, w;
  int64_t N;
  float* X; float* zin; float* deformed; const float* dX; float* fpart;
  int64_t chunk; int O;
  float* dgrid;   // backward, single object (optional): d / d grid, planar [B][2][H][W]
};

// arena block of one backbone: [b1 (w) | g1 | v1 (w) | b2 | g2 | v2 (w)]
__device__ __forceinline__ int bb_size(int w) { return 3 * w + 3; }
// effective block in shared memory: [w1 (w) | b1 (w) | w2 (w) | b2]
__device__ __forceinline__ int eff_size(int w) { return 3 * w + 1; }

// Stage effective weights: eff[(2*i + which) * eff_size] for coupling i, which = 0 (S) / 1 (T); cs[i] = c_i;
// lin[0..3] = W (row major), lin[4..5] = bias.
__device__ void stage_effective(const DiffP& p, const float* par, float* eff, float* cs, float* lin, float* norms) {
  const int w = p.w, nc = p.nc, bs = bb_size(w), es = eff_size(w);
  // norms[(2*i + which) * 2 + layer] = ||v||
  for (int t = threadIdx.x; t < nc * 4; t += blockDim.x) {
    const int i = t >> 2, which = (t >> 1) & 1, layer = t & 1;
    const float* blk = par + (int64_t)(which * nc + i) * bs;
    const float* v = layer == 0 ? blk + w + 1 : blk + 2 * w + 3;
    float a = 0.f;
    for (int k = 0; k < w; k++) a = fmaf(v[k], v[k], a);
    norms[t] = sqrtf(a);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < nc * 2 * w; t += blockDim.x) {
    const int k = t % w, bi = t / w, i = bi >> 1, which = bi & 1;
    const float* blk = par + (int64_t)(which * nc + i) * bs;
    float* e = eff + (int64_t)bi * es;
    e[k] = blk[w] * blk[w + 1 + k] / norms[bi * 2];                 // w1 = g1 * v1 / ||v1||
    e[w + k] = blk[k];                                             // b1
    e[2 * w + k] = blk[2 * w + 2] * blk[2 * w + 3 + k] / norms[bi * 2 + 1];   // w2
    if (k == 0) e[3 * w] = blk[2 * w + 1];                         // b2
  }
  if (threadIdx.x < nc) {
    const float* sc = par + (int64_t)2 * nc * bs + threadIdx.x * 4;          // [weight, bias, g, v]
    const float sgn = sc[3] > 0.f ? 1.f : (sc[3] < 0.f ? -1.f : 0.f);
    cs[threadIdx.x] = fmaf(sc[2] * sgn, sc[0], sc[1]);
  }
  if (threadIdx.x < 6) lin[threadIdx.x] = par[(int64_t)2 * nc * bs + 4 * nc + threadIdx.x];
  __syncthreads();
}

__global__ void __launch_bounds__(256) k_diffeo_fwd(DiffP p) {
  extern __shared__ float sm[];
  const int w = p.w, nc = p.nc, es = eff_size(w);
  float* eff = sm;
  float* cs = eff + nc * 2 * es;
  float* lin = cs + kMaxNC;
  float* norms = lin + 8;
  const int o = blockIdx.y;
  stage_effective(p, p.params + (int64_t)o * p.P + p.off_flow, eff, cs, lin, norms);
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.N) return;
  const float gx = coord(p.g, n, 0), gy = coord(p.g, n, 1);
  float x1 = fmaf(lin[0], gx, fmaf(lin[1], gy, lin[4]));
  float x2 = fmaf(lin[2], gx, fmaf(lin[3], gy, lin[5]));
  float* zin = p.zin ? p.zin + ((int64_t)o * p.N + n) * (nc * 2) : nullptr;
  for (int i = 0; i < nc; i++) {
    if (zin) { zin[2 * i] = x1; zin[2 * i + 1] = x2; }
    const float in = (i & 1) ? x2 : x1;
    const float* es_ = eff + (int64_t)(2 * i) * es;
    const float* et_ = es_ + es;
    float ss = es_[3 * w], tt = et_[3 * w];
    for (int k = 0; k < w; k++) {
      ss = fmaf(es_[2 * w + k], fmaxf(fmaf(es_[k], in, es_[w + k]), 0.f), ss);
      tt = fmaf(et_[2 * w + k], fmaxf(fmaf(et_[k], in, et_[w + k]), 0.f), tt);
    }
    const float hs = tanhf(ss), ht = tanhf(tt);
    if (i & 1) x1 = fmaf(expf(cs[i] * hs), x1, ht);
    else x2 = fmaf(expf(cs[i] * hs), x2, ht);
  }
  *reinterpret_cast<float4*>(p.X + ((int64_t)o * p.N + n) * 4) = make_float4(x1, x2, 0.f, 1.f);
  if (p.deformed) { p.deformed[((int64_t)o * p.N + n) * 2] = x1; p.deformed[((int64_t)o * p.N + n) * 2 + 1] = x2; }
}

// DG: also write the coordinate gradient p.dgrid (a separate instantiation, so that the fit path's code is untouched)
template <int NC, bool DG>
__global__ void __launch_bounds__(256) k_diffeo_bwd(DiffP p) {
  extern __shared__ float sm[];
  const int w = p.w, es = eff_size(w), bs = bb_size(w);
  float* eff = sm;
  float* cs = eff + NC * 2 * es;
  float* lin = cs + kMaxNC;
  float* norms = lin + 8;
  float* red = norms + 8 * kMaxNC;          // [8 warps][RED] per-warp sums, then the CTA totals in red[0..RED)
  const int RED = NC * 2 * 3 * w + NC * 3 + 6;   // unit arrays (w1, b1, w2 per backbone) | per coupling (b2s, b2t, c) | linear
  const int o = blockIdx.y, s = blockIdx.x;
  const float* par = p.params + (int64_t)o * p.P + p.off_flow;
  stage_effective(p, par, eff, cs, lin, norms);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float gw1[NC][2][3], gb1[NC][2][3], gw2[NC][2][3], gsc[NC][3], glin[6];
#pragma unroll
  for (int i = 0; i < NC; i++) {
#pragma unroll
    for (int b = 0; b < 2; b++)
#pragma unroll
      for (int u = 0; u < 3; u++) { gw1[i][b][u] = 0.f; gb1[i][b][u] = 0.f; gw2[i][b][u] = 0.f; }
    gsc[i][0] = gsc[i][1] = gsc[i][2] = 0.f;
  }
#pragma unroll
  for (int i = 0; i < 6; i++) glin[i] = 0.f;
  const int64_t r0 = (int64_t)s * p.chunk, r1 = r0 + p.chunk < p.N ? r0 + p.chunk : p.N;
  for (int64_t n = r0 + warp; n < r1; n += nw) {
    const float* dx = p.dX + ((int64_t)o * p.N + n) * 4;
    float dz1 = dx[0], dz2 = dx[1];
    const float* zin = p.zin + ((int64_t)o * p.N + n) * (NC * 2);
#pragma unroll
    for (int i = NC - 1; i >= 0; i--) {
      const float x1 = zin[2 * i], x2 = zin[2 * i + 1];
      const float in = (i & 1) ? x2 : x1, tv = (i & 1) ? x1 : x2, dout = (i & 1) ? dz1 : dz2;
      float pre[2][3], hh[2][3], acc[2] = {0.f, 0.f};
#pragma unroll
      for (int b = 0; b < 2; b++) {
        const float* e = eff + (int64_t)(2 * i + b) * es;
#pragma unroll
        for (int u = 0; u < 3; u++) {
          const int k = lane + 32 * u;
          pre[b][u] = k < w ? fmaf(e[k], in, e[w + k]) : 0.f;
          hh[b][u] = fmaxf(pre[b][u], 0.f);
          if (k < w) acc[b] = fmaf(e[2 * w + k], hh[b][u], acc[b]);
        }
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], off);
        acc[1] += __shfl_xor_sync(0xffffffffu, acc[1], off);
      }
      const float hs = tanhf(acc[0] + eff[(int64_t)(2 * i) * es + 3 * w]);
      const float ht = tanhf(acc[1] + eff[(int64_t)(2 * i + 1) * es + 3 * w]);
      const float c = cs[i], ex = expf(c * hs);
      const float d_e = dout * tv;
      const float d_hs = d_e * ex * c;
      gsc[i][2] = fmaf(d_e * ex, hs, gsc[i][2]);                       // d c_i
      const float dpre[2] = {d_hs * (1.f - hs * hs), dout * (1.f - ht * ht)};
      gsc[i][0] += dpre[0]; gsc[i][1] += dpre[1];                       // d b2 of S, T
      float din = 0.f;
#pragma unroll
      for (int b = 0; b < 2; b++) {
        const float* e = eff + (int64_t)(2 * i + b) * es;
#pragma unroll
        for (int u = 0; u < 3; u++) {
          const int k = lane + 32 * u;
          if (k < w) {
            gw2[i][b][u] = fmaf(dpre[b], hh[b][u], gw2[i][b][u]);
            const float dh = pre[b][u] > 0.f ? dpre[b] * e[2 * w + k] : 0.f;
            gw1[i][b][u] = fmaf(dh, in, gw1[i][b][u]);
            gb1[i][b][u] += dh;
            din = fmaf(dh, e[k], din);
          }
        }
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) din += __shfl_xor_sync(0xffffffffu, din, off);
      if (i & 1) { dz1 = dout * ex; dz2 += din; } else { dz2 = dout * ex; dz1 += din; }
    }
    const float gx = coord(p.g, n, 0), gy = coord(p.g, n, 1);
    glin[0] = fmaf(dz1, gx, glin[0]); glin[1] = fmaf(dz1, gy, glin[1]);
    glin[2] = fmaf(dz2, gx, glin[2]); glin[3] = fmaf(dz2, gy, glin[3]);
    glin[4] += dz1; glin[5] += dz2;
    if (DG && lane == 0) {          // coordinate gradient W^T (dz1, dz2): every lane holds the same dz1, dz2
      p.dgrid[planar_index(p.g, n, 0)] = fmaf(lin[0], dz1, lin[2] * dz2);
      p.dgrid[planar_index(p.g, n, 1)] = fmaf(lin[1], dz1, lin[3] * dz2);
    }
  }
  // ---- per-warp sums -> shared memory -> fixed-order sum over the warps
  float* mine = red + (int64_t)warp * RED;
#pragma unroll
  for (int i = 0; i < NC; i++)
#pragma unroll
    for (int b = 0; b < 2; b++)
#pragma unroll
      for (int u = 0; u < 3; u++) {
        const int k = lane + 32 * u;
        if (k < w) {
          float* q = mine + (int64_t)((2 * i + b) * 3) * w;
          q[k] = gw1[i][b][u]; q[w + k] = gb1[i][b][u]; q[2 * w + k] = gw2[i][b][u];
        }
      }
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NC; i++) { mine[NC * 6 * w + 3 * i] = gsc[i][0]; mine[NC * 6 * w + 3 * i + 1] = gsc[i][1]; mine[NC * 6 * w + 3 * i + 2] = gsc[i][2]; }
#pragma unroll
    for (int i = 0; i < 6; i++) mine[NC * 6 * w + 3 * NC + i] = glin[i];
  }
  __syncthreads();
  for (int t = threadIdx.x; t < RED; t += blockDim.x) {
    float a = 0.f;
    for (int ww = 0; ww < nw; ww++) a += red[(int64_t)ww * RED + t];
    red[t] = a;     // (ww = 0 row is read before it is overwritten by this same thread)
  }
  __syncthreads();
  // ---- weight-norm Jacobian: effective-weight gradients -> (bias, g, v) gradients in state_dict order
  float* out = p.fpart + ((int64_t)s * p.O + o) * p.PF;
  float* dots = norms + 4 * NC;             // [NC*4] sum_k dW[k] * v[k] / ||v||
  for (int t = threadIdx.x; t < NC * 4; t += blockDim.x) {
    const int i = t >> 2, which = (t >> 1) & 1, layer = t & 1;
    const float* blk = par + (int64_t)(which * NC + i) * bs;
    const float* v = layer == 0 ? blk + w + 1 : blk + 2 * w + 3;
    const float* dw = red + (int64_t)((2 * i + which) * 3 + (layer == 0 ? 0 : 2)) * w;
    float a = 0.f;
    for (int k = 0; k < w; k++) a = fmaf(dw[k], v[k], a);
    dots[t] = a / norms[(2 * i + which) * 2 + layer];
  }
  __syncthreads();
  for (int t = threadIdx.x; t < NC * 2 * w; t += blockDim.x) {
    const int k = t % w, bi = t / w, i = bi >> 1, which = bi & 1;
    const float* blk = par + (int64_t)(which * NC + i) * bs;
    float* ob = out + (int64_t)(which * NC + i) * bs;
    const float* q = red + (int64_t)(bi * 3) * w;
    const float n1 = norms[bi * 2], n2 = norms[bi * 2 + 1], g1 = blk[w], g2 = blk[2 * w + 2];
    const int t1 = (i << 2) | (which << 1), t2 = t1 | 1;
    ob[k] = q[w + k];                                                                  // d b1
    ob[w + 1 + k] = g1 / n1 * (q[k] - dots[t1] * blk[w + 1 + k] / n1);                   // d v1
    ob[2 * w + 3 + k] = g2 / n2 * (q[2 * w + k] - dots[t2] * blk[2 * w + 3 + k] / n2);   // d v2
    if (k == 0) {
      ob[w] = dots[t1];                                                                // d g1
      ob[2 * w + 2] = dots[t2];                                                        // d g2
      ob[2 * w + 1] = red[NC * 6 * w + 3 * i + which];                                 // d b2
    }
  }
  if (threadIdx.x < NC) {
    const int i = threadIdx.x;
    const float* sc = par + (int64_t)2 * NC * bs + i * 4;
    float* os = out + (int64_t)2 * NC * bs + i * 4;
    const float sgn = sc[3] > 0.f ? 1.f : (sc[3] < 0.f ? -1.f : 0.f);
    const float gc = red[NC * 6 * w + 3 * i + 2];
    os[0] = gc * sc[2] * sgn;      // d weight
    os[1] = gc;                    // d scale.bias
    os[2] = gc * sc[0] * sgn;      // d scale.weight_g
    os[3] = 0.f;                   // d scale.weight_v: v / |v| is locally constant for a 1x1 weight
  }
  if (threadIdx.x < 6) out[(int64_t)2 * NC * bs + 4 * NC + threadIdx.x] = red[NC * 6 * w + 3 * NC + threadIdx.x];
}

// ======================================================================= launchers
static DiffP make_dp(const awb_prior* h, const float* params, const awb_grid_spec* g, const Workspace& ws) {
  const Layout& L = h->lay;
  DiffP p = {};
  p.g.mode = g->mode; p.g.B = g->B; p.g.H = g->H; p.g.W = g->W; p.g.C = L.C; p.g.t0 = g->t0; p.g.t_step = g->t_step; p.g.grid = g->grid;
  p.params = params; p.P = L.P; p.off_flow = L.off_flow; p.PF = L.P_flow + L.n_lin;
  p.nc = L.F; p.w = L.m;
  p.N = (int64_t)g->B * g->H * g->W;
  p.X = ws.X; p.zin = nullptr; p.deformed = nullptr; p.dX = ws.dX; p.fpart = ws.fpart;
  p.chunk = split_chunk(p.N); p.O = h->desc.n_objects; p.dgrid = nullptr;
  return p;
}

int diffeo_forward(const awb_prior* h, const float* params, const awb_grid_spec* g, const Workspace& ws, float* deformed,
                   cudaStream_t st) {
  DiffP p = make_dp(h, params, g, ws);
  p.zin = ws.flowz;
  p.deformed = deformed;
  const size_t smem = sizeof(float) * ((size_t)p.nc * 2 * (3 * p.w + 1) + kMaxNC + 8 + 8 * kMaxNC);
  dim3 grid((unsigned)((p.N + 255) / 256), h->desc.n_objects);
  AWB_LAUNCH(PK_FLOW_FWD, st, k_diffeo_fwd<<<grid, 256, smem, st>>>(p));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int diffeo_backward(const awb_prior* h, const float* params, const awb_grid_spec* g, const Workspace& ws, cudaStream_t st,
                    float* dgrid) {
  DiffP p = make_dp(h, params, g, ws);
  p.zin = ws.flowz;
  p.dgrid = dgrid;
  if (!p.zin) { set_error("flow backward needs a training workspace"); return AWB_ERR_WORKSPACE; }
  if (dgrid && h->desc.n_objects != 1) { set_error("internal: dgrid needs one object"); return AWB_ERR_INVALID; }
  const int RED = p.nc * 2 * 3 * p.w + p.nc * 3 + 6;
  const size_t smem = sizeof(float) * ((size_t)p.nc * 2 * (3 * p.w + 1) + kMaxNC + 8 + 8 * kMaxNC + 8 * (size_t)RED);
  dim3 grid(n_splits(p.N), h->desc.n_objects);
#define AWB_DIFFEO_BWD(NC_)                                                                                    \
  do {                                                                                                         \
    auto kernel = p.dgrid ? k_diffeo_bwd<NC_, true> : k_diffeo_bwd<NC_, false>;                              \
    AWB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));           \
    AWB_LAUNCH(PK_FLOW_BWD, st, kernel<<<grid, 256, smem, st>>>(p));                                          \
  } while (0)
  if (p.nc == 2) AWB_DIFFEO_BWD(2);
  else if (p.nc == 4) AWB_DIFFEO_BWD(4);
  else if (p.nc == 6) AWB_DIFFEO_BWD(6);
  else if (p.nc == 8) AWB_DIFFEO_BWD(8);
  else { set_error("NormalizingFlow1D: num_coupling must be 2, 4, 6 or 8, got %d", p.nc); return AWB_ERR_UNSUPPORTED; }
#undef AWB_DIFFEO_BWD
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

}  // namespace awb
