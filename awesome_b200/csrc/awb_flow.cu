// RealNVP path-connectedness flow (SURVEY a2/a3/a5): grouped 1x1 conv on the coordinates
// (path_connected_net.py:65,82), MinMax to [-1,1] (min_max.py:9-19, norm_net.py:17-27), F x
// { MaskedAffineFlow(b, t, s); ActNorm } with s,t = MLP([C,m,C], LeakyReLU(0), tanh) (normflows
// 1.7.3 published semantics, see DESIGN.md; built at net_factory.py:101-113), inverse
// MinMax.  K = C = 2..3 is too thin for tensor cores: CUDA-core FMAs, everything per pixel stays in
// registers, weights are staged once per CTA in shared memory.
//
// forward : four pixels per thread (no cross-pixel reduction).  Writes the deformed coordinates
//           X[n] = (x, y, t, 1) consumed by the ICNN and, when training, the input and the (s, t) outputs of every
//           coupling (4 / 8 floats per pixel and flow) so that the backward pass needs no forward sweep.
// backward: ONE kernel (k_flow_bwd): a CTA owns a pixel range, keeps the running coordinate gradient in shared memory and
//           walks the flows in reverse; per hidden unit it accumulates in registers the masked sums every weight gradient
//           is linear in.  No atomics, no per-pixel record through global memory; partials are reduced in a fixed order.
#include <math.h>

#include <type_traits>

#include "awb_internal.cuh"

namespace awb {

struct FlowP {
  GridDev g;
  FlowConsts fc;
  const float* params;   // arena, object 0
  int64_t P, off_flow, P_flow, per_flow, off_lin;
  int C, F, m, tanh_out, use_linear;
  float out_scale;       // normflows MLP output_scale: s, t = out_scale * tanh(.) (1 when unset; only with an output_fn)
  float inv_out_scale;
  int64_t N;
  float* X;              // [O][N][4]
  float* zin;            // [O][F][N][RW] saved coupling inputs / outputs (FlowSave), or null
  float* deformed;       // [O][N][C] or null
  float* dX;             // backward: [O][N][4] (overwritten in place when the range does not fit in shared memory)
  float* fpart;          // backward: [S][O][PF]
  int64_t chunk; int O;
  int rounds;            // rounds of FLOW_P / FLOW_PB pixels per thread
  int rounds1;           // backward: remainder rounds of one pixel per thread
  int dz_smem;           // backward: the running coordinate gradient of the CTA's pixel range lives in shared memory
  float* dzp_g;          // backward, C = 3, !dz_smem: [O][N][4] scratch for the partial gradient between unit passes
  float* tab;            // C = 2: [O][F][FLOW_TAB] segment tables of the coupling MLPs (k_flow_tables), or null
  float* segscr;         // C = 2 backward: [S][O][F][8 warps][FLOW_SEG_RS] per-warp histogram sums
  float* dgrid;          // backward, single object (optional): d / d grid, planar [B][C][H][W]
};

// tanh and exp of the coupling outputs on the special-function unit: tanh(a) = 1 - 2 / (exp(2a) + 1) with ex2.approx /
// rcp.approx (absolute error <= 2e-7, exact at a = 0 where the zero-initialised couplings start, saturates to +-1, NaN
// propagates), exp of s in [-1, 1] with ex2.approx (relative error <= 2e-7) -- 6 + 2 instructions instead of ~35 + 8 of
// tanhf / expf.  The inverse and the ActNorm init keep the library functions.
__device__ __forceinline__ float tanh_sfu(float a) { return 1.f - __fdividef(2.f, __expf(2.f * a) + 1.f); }
__device__ __forceinline__ float exp_sfu(float s) { return __expf(s); }

__device__ __forceinline__ float mm_fwd(float v, float vmin, float vmax, float nmin, float nmax) {
  // (v - min) / (max - min) * (new_max - new_min) + new_min, in the reference's order (min_max.py:9-19).  A span of exactly 1
  // (the [0, 1] coordinate grid every config normalises from / to) divides exactly: the IEEE division (~25 instructions, four
  // per pixel) is skipped without changing a bit.
  const float d = vmax - vmin, x = v - vmin;
  return (d == 1.f ? x : x / d) * (nmax - nmin) + nmin;
}

// ---- k-packed weight staging for the per-pixel kernels.  The MLP loops read, per hidden unit k, the 4C+2 scalars
// (w1s[C], b1s, w2s[C], w1t[C], b1t, w2t[C]); in state_dict order they sit in 6 different arrays (6 broadcast LDS per
// unit).  Staged as one padded record per (flow, unit) they are 3 (C=2) / 4 (C=3) LDS.128 -- the loops are
// shared-memory-issue bound, not FMA bound.  Per flow: [m records | b2s[C] | b2t[C] | an_s[C] | an_t[C]].
template <int C> struct FlowPack {
  static constexpr int RK = (4 * C + 2 + 3) / 4 * 4;       // 12 (C=2), 16 (C=3)
  __host__ __device__ static int flow_stride(int m) { return m * RK + 4 * C; }
};
// Flows whose mask pattern is one of the compiled-in ones (binary codes 1 .. 2^C - 2) get a COMPACT record in the first 8
// floats: only what the pattern uses -- [w1s of the masked comps | b1s | w2s of the transformed comps | w1t masked | b1t |
// w2t transformed] = 2C + 2 <= 8 floats = 2 LDS.128 per hidden unit instead of 3 (C = 2) / 4 (C = 3).
template <int C>
__device__ __forceinline__ bool flow_pattern_compiled(int mb) { return mb >= 1 && mb <= (1 << C) - 2; }
template <int C>
__device__ void stage_flow_packed(const float* __restrict__ par, int F, int m, int64_t per_flow, float* sp, const FlowConsts& fc,
                                  bool exp_actnorm = false) {
  constexpr int RK = FlowPack<C>::RK;
  const int half = 2 * m * C + m + C, FS = FlowPack<C>::flow_stride(m);
  for (int t = threadIdx.x; t < F * m; t += blockDim.x) {
    const int f = t / m, k = t - f * m;
    const float* w = par + (int64_t)f * per_flow;
    float* r = sp + f * FS + k * RK;
    int mb = 0;
#pragma unroll
    for (int c = 0; c < C; c++) mb |= fc.masks[f * C + c] != 0 ? 1 << c : 0;
    if (flow_pattern_compiled<C>(mb)) {
      int pos = 0;
      for (int c = 0; c < C; c++) if ((mb >> c) & 1) r[pos++] = w[k * C + c];                              // s.W1[k][c], masked c
      r[pos++] = w[m * C + k];                                                                         // s.b1[k]
      for (int c = 0; c < C; c++) if (!((mb >> c) & 1)) r[pos++] = w[m * C + m + c * m + k];               // s.W2[c][k], transformed c
      for (int c = 0; c < C; c++) if ((mb >> c) & 1) r[pos++] = w[half + k * C + c];                       // t.W1[k][c]
      r[pos++] = w[half + m * C + k];                                                                  // t.b1[k]
      for (int c = 0; c < C; c++) if (!((mb >> c) & 1)) r[pos++] = w[half + m * C + m + c * m + k];        // t.W2[c][k]
      continue;
    }
#pragma unroll
    for (int c = 0; c < C; c++) {
      r[c] = w[k * C + c];                               // s.W1[k][c]
      r[C + 1 + c] = w[m * C + m + c * m + k];           // s.W2[c][k]
      r[2 * C + 1 + c] = w[half + k * C + c];            // t.W1[k][c]
      r[3 * C + 2 + c] = w[half + m * C + m + c * m + k];   // t.W2[c][k]
    }
    r[C] = w[m * C + k];                                 // s.b1[k]
    r[3 * C + 1] = w[half + m * C + k];                  // t.b1[k]
  }
  for (int t = threadIdx.x; t < F * 4 * C; t += blockDim.x) {
    const int f = t / (4 * C), j = t - f * 4 * C, q = j / C, c = j - q * C;
    const float* w = par + (int64_t)f * per_flow;
    const float v = q == 0 ? w[m * C + m + C * m + c] : q == 1 ? w[half + m * C + m + C * m + c] : w[2 * half + (q - 2) * C + c];
    sp[f * FS + m * RK + j] = (exp_actnorm && q == 2) ? expf(v) : v;
  }
}


// ---- coupling MLPs with the mask pattern of the flow known at compile time.  MB: bit c set = component c is masked
// (passes through the coupling and feeds s / t); MB < 0 = pattern only known at run time.  With the pattern fixed, the
// multiplications by a masked-out zero and the outputs nobody reads disappear (half of the FMAs for the alternating
// masks of net_factory.py:86-99); the surviving arithmetic is unchanged, so results are bit-identical.
template <int C, int MB>
__device__ __forceinline__ bool masked_c(int c, const bool* b) { return MB < 0 ? b[c] : ((MB >> c) & 1) != 0; }

// s / t pre-outputs of one coupling: so[c], to[c] for the transformed components (the others are left untouched)
// record of hidden unit k: compact (8 floats) for a compiled-in pattern, the full RK floats otherwise
template <int C, int MB>
struct FlowRec {
  static constexpr int NM = MB < 0 ? 0 : ((MB & 1) + ((MB >> 1) & 1) + ((MB >> 2) & 1));     // masked components
  static constexpr int NU = C - NM;
  static constexpr int N4 = MB < 0 ? FlowPack<C>::RK / 4 : 2;
  float v[4 * N4];
  __device__ __forceinline__ void load(const float* __restrict__ rec) {
#pragma unroll
    for (int q4 = 0; q4 < N4; q4++) *reinterpret_cast<float4*>(&v[4 * q4]) = reinterpret_cast<const float4*>(rec)[q4];
  }
  // rank of component c among the masked / the transformed ones (constant-folded after unrolling)
  static __device__ __forceinline__ int rm(int c) { return __popc(MB & ((1 << c) - 1)); }
  static __device__ __forceinline__ int ru(int c) { return c - rm(c); }
  __device__ __forceinline__ float w1s(int c) const { return MB < 0 ? v[c] : v[rm(c)]; }
  __device__ __forceinline__ float b1s() const { return MB < 0 ? v[C] : v[NM]; }
  __device__ __forceinline__ float w2s(int c) const { return MB < 0 ? v[C + 1 + c] : v[NM + 1 + ru(c)]; }
  __device__ __forceinline__ float w1t(int c) const { return MB < 0 ? v[2 * C + 1 + c] : v[NM + 1 + NU + rm(c)]; }
  __device__ __forceinline__ float b1t() const { return MB < 0 ? v[3 * C + 1] : v[2 * NM + 1 + NU]; }
  __device__ __forceinline__ float w2t(int c) const { return MB < 0 ? v[3 * C + 2 + c] : v[2 * NM + 2 + NU + ru(c)]; }
};

// P pixels per thread share every weight record: the per-pixel kernels are bound by the shared-memory loads of the
// records (2 LDS.128 per ~6 FMAs with one pixel), not by the FMAs.
template <int C, int MB, int P>
__device__ __forceinline__ void coupling_mlp_fwd(const float* __restrict__ wf, int m, const float (*z)[C], const bool* b,
                                                 float (*so)[C], float (*to)[C]) {
  constexpr int RK = FlowPack<C>::RK;
#pragma unroll 4
  for (int k = 0; k < m; k++) {
    FlowRec<C, MB> r;
    r.load(wf + k * RK);
#pragma unroll
    for (int q = 0; q < P; q++) {
      float ps = r.b1s(), pt = r.b1t();
#pragma unroll
      for (int c = 0; c < C; c++)
        if (masked_c<C, MB>(c, b)) { ps = fmaf(r.w1s(c), z[q][c], ps); pt = fmaf(r.w1t(c), z[q][c], pt); }
      const float hs = fmaxf(ps, 0.f), ht = fmaxf(pt, 0.f);
#pragma unroll
      for (int c = 0; c < C; c++)
        if (MB < 0 || !masked_c<C, MB>(c, b)) {
          so[q][c] = fmaf(r.w2s(c), hs, so[q][c]);
          to[q][c] = fmaf(r.w2t(c), ht, to[q][c]);
        }
    }
  }
}

// warp-uniform dispatch on the flow's mask pattern: every pattern net_factory.py:86-99 produces (the binary codes
// 1 .. 2^C - 2) is compiled in for C = 2 and C = 3; anything else runs the generic path
#define AWB_FLOW_DISPATCH(C_, mb_, CALL)                                  \
  do {                                                                    \
    if ((mb_) == 1) { CALL(1); }                                          \
    else if ((mb_) == 2) { CALL(2); }                                     \
    else if ((C_) == 3 && (mb_) == 3) { CALL(3); }                        \
    else if ((C_) == 3 && (mb_) == 4) { CALL(4); }                        \
    else if ((C_) == 3 && (mb_) == 5) { CALL(5); }                        \
    else if ((C_) == 3 && (mb_) == 6) { CALL(6); }                        \
    else { CALL(-1); }                                                    \
  } while (0)

// ---- launch geometry of the forward and the backward kernel: S pixel ranges of `chunk` rows (one CTA each, per
// object), T threads per CTA, R full rounds of P pixels per thread, then the remainder of the range in rounds of one
// pixel per thread.  Pixel of (slot q, thread t) of a round starting at `base` = base + q * T + t: consecutive threads
// touch consecutive pixels (coalesced).
struct FlowGeo { int S, T, R; int64_t chunk; };
// Saved per pixel and flow for the backward pass (training forward): the coupling's input z[C] and the post-activation
// outputs s, t of its two MLPs for the transformed components -- RW floats, stored [O][F][N][RW] (pixel-contiguous:
// full-sector vector stores / loads).  C = 2: (z0, z1, s, t); C = 3: (z0, z1, z2, s_a | s_b, t_a, t_b, -) with a, b the
// transformed components in ascending order.
template <int C> struct FlowSave { static constexpr int RW = C == 2 ? 4 : 8; };
int flow_save_floats(int C) { return C == 2 ? 4 : 8; }

constexpr int FLOW_TAB3 = 584;     // C = 3 forward tables, see k_flow_tables3
// number of merged breakpoints below z (0 .. 64) TIMES 4: lower bound over gamma[0..62] in six dependent steps, gamma[63] on
// its own.  `tab`: shared-space address of the table (ld.shared with an immediate offset per step: load, compare,
// predicated add).
__device__ __forceinline__ float lds_f32(uint32_t a) { float v; asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) { uint32_t v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ float2 lds_f32x2(uint32_t a) { float2 v; asm("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a)); return v; }
__device__ __forceinline__ float4 lds_f32x4(uint32_t a) {
  float4 v;
  asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
// the same for PP pixels at once, breadth first (step k of every pixel before step k + 1 of any): the PP dependent chains
// of loads overlap instead of running one after the other
template <int PP>
__device__ __forceinline__ void seg_find4_multi(uint32_t tab, const float* z, uint32_t* o) {
  const float g31 = lds_f32(tab + 31 * 4), g63 = lds_f32(tab + 63 * 4);
  uint32_t top[PP];
#pragma unroll
  for (int q = 0; q < PP; q++) { o[q] = g31 < z[q] ? 128u : 0u; top[q] = g63 < z[q] ? 4u : 0u; }
#pragma unroll
  for (int k = 0; k < 5; k++) {
    const uint32_t off = (15u >> k) * 4u, inc = 64u >> k;      // (15, 64), (7, 32), (3, 16), (1, 8), (0, 4)
    float v[PP];
#pragma unroll
    for (int q = 0; q < PP; q++) v[q] = lds_f32(tab + o[q] + off);
#pragma unroll
    for (int q = 0; q < PP; q++) o[q] += v[q] < z[q] ? inc : 0u;
  }
#pragma unroll
  for (int q = 0; q < PP; q++) o[q] += top[q];
}
__device__ __forceinline__ uint32_t seg_find4(uint32_t tab, float z) {
  uint32_t o = lds_f32(tab + 31 * 4) < z ? 128u : 0u;
  const uint32_t top = lds_f32(tab + 63 * 4) < z ? 4u : 0u;
  o += lds_f32(tab + o + 15 * 4) < z ? 64u : 0u;
  o += lds_f32(tab + o + 7 * 4) < z ? 32u : 0u;
  o += lds_f32(tab + o + 3 * 4) < z ? 16u : 0u;
  o += lds_f32(tab + o + 1 * 4) < z ? 8u : 0u;
  o += lds_f32(tab + o) < z ? 4u : 0u;
  return o + top;
}

constexpr int FLOW_P = 4;          // forward: pixels per thread and round: every weight record (2-3 LDS.128) feeds 4 pixels
constexpr int FLOW_PB = 4;         // backward: same, bounded by the 128 accumulator registers beside them
constexpr int FLOW_RED_FLOATS = 16 * 128 + 16 * 16;   // one reduction scratch: 16 warps x (128 accumulator sums + 16 scalar sums)
constexpr int FLOW_BWD_T = 256;    // 8 warps = 2 per scheduler: up to 255 registers per thread
template <int C>
__global__ void __launch_bounds__(256) k_flow_fwd(FlowP p) {
  extern __shared__ __align__(16) float sp[];   // k-packed flow weights + [2C] linear
  constexpr int RK = FlowPack<C>::RK;
  constexpr int RW = FlowSave<C>::RW;
  const int o = blockIdx.y;
  const float* par = p.params + (int64_t)o * p.P + p.off_flow;
  const int m = p.m, FS = FlowPack<C>::flow_stride(m);
  stage_flow_packed<C>(par, p.F, m, p.per_flow, sp, p.fc, /*exp_actnorm=*/true);
  float* lin = sp + p.F * FS;
  if (threadIdx.x < 2 * C) lin[threadIdx.x] = par[p.P_flow + threadIdx.x];
  // C = 3 on the tensor path: segment tables of the flows with one masked coordinate behind the weights (k_flow_tables3)
  const bool seg3 = C == 3 && p.tab != nullptr;
  float* tab3 = lin + 2 * C + 2;          // 16-byte aligned: F * FS and 2 C + 2 are multiples of 4 floats
  if (seg3) {
    const float* tg = p.tab + (int64_t)o * p.F * FLOW_TAB3;
    for (int i = threadIdx.x; i < p.F * (FLOW_TAB3 / 4); i += blockDim.x) {
      const int f = i / (FLOW_TAB3 / 4);
      int mbf = 0;
#pragma unroll
      for (int c = 0; c < C; c++) mbf |= p.fc.masks[f * C + c] != 0 ? 1 << c : 0;
      if (__popc(mbf) == 1) reinterpret_cast<float4*>(tab3)[i] = reinterpret_cast<const float4*>(tg)[i];
    }
  }
  __syncthreads();
  const int T = blockDim.x;
  const int64_t r0 = (int64_t)blockIdx.x * p.chunk, r1 = r0 + p.chunk < p.N ? r0 + p.chunk : p.N;
  // one round: P pixels of this thread starting at `base` (slot q -> pixel base + q * T + tid) share every weight record
  auto round = [&](auto p_c, int64_t base) -> bool {
    constexpr int P = decltype(p_c)::value;
    int64_t n[P];
    bool ok[P];
    float z[P][C];
#pragma unroll
    for (int q = 0; q < P; q++) {
      const int64_t nq = base + (int64_t)q * T + threadIdx.x;
      ok[q] = nq < r1;
      n[q] = ok[q] ? nq : (r1 > 0 ? r1 - 1 : 0);          // padding slots recompute the range's last pixel and store nothing
#pragma unroll
      for (int c = 0; c < C; c++) {
        float x = coord(p.g, n[q], c);
        if (p.use_linear) x = x * lin[c] + lin[C + c];
        z[q][c] = mm_fwd(x, p.fc.nmin[c], p.fc.nmax[c], p.fc.new_min, p.fc.new_max);
      }
    }
    if (!ok[0]) return false;
    for (int f = 0; f < p.F; f++) {
      const float* wf = sp + f * FS;
      const float* tail = wf + m * RK;          // b2s[C] | b2t[C] | exp(an_s)[C] | an_t[C]
      bool b[C];
      int mb = 0;
#pragma unroll
      for (int c = 0; c < C; c++) { b[c] = p.fc.masks[f * C + c] != 0; mb |= b[c] ? 1 << c : 0; }
      float so[P][C], to[P][C];
#pragma unroll
      for (int q = 0; q < P; q++) {
#pragma unroll
        for (int c = 0; c < C; c++) { so[q][c] = tail[c]; to[q][c] = tail[C + c]; }
      }
      if (C == 3 && seg3 && (mb == 1 || mb == 2 || mb == 4)) {
        // one masked coordinate: both MLPs are piecewise linear in it -- one search over the merged breakpoints and one FMA
        // per net and output instead of the unit loop (same pre-activation outputs up to the order of the sums)
        const uint32_t tb = (uint32_t)__cvta_generic_to_shared(tab3 + f * FLOW_TAB3);
        auto seg_couple = [&](auto cm_c) {
          constexpr int cm = decltype(cm_c)::value < C ? decltype(cm_c)::value : 0;
          constexpr int ua = cm == 0 ? 1 : 0, ub = cm == C - 1 ? C - 2 : C - 1;
          float zm[P];
          uint32_t J4[P];
#pragma unroll
          for (int q = 0; q < P; q++) zm[q] = z[q][cm];
          seg_find4_multi<P>(tb, zm, J4);
#pragma unroll
          for (int q = 0; q < P; q++) {
            const float4 sl = lds_f32x4(tb + 256 + 8 * J4[q]), ic = lds_f32x4(tb + 256 + 8 * J4[q] + 16);
            so[q][ua] = fmaf(sl.x, zm[q], ic.x); so[q][ub] = fmaf(sl.y, zm[q], ic.y);
            to[q][ua] = fmaf(sl.z, zm[q], ic.z); to[q][ub] = fmaf(sl.w, zm[q], ic.w);
          }
        };
        if (mb == 1) seg_couple(std::integral_constant<int, 0>{});
        else if (mb == 2) seg_couple(std::integral_constant<int, 1>{});
        else seg_couple(std::integral_constant<int, 2>{});
      } else {
#define AWB_CALL(MB) coupling_mlp_fwd<C, MB, P>(wf, m, z, b, so, to)
        AWB_FLOW_DISPATCH(C, mb, AWB_CALL);
#undef AWB_CALL
      }
#pragma unroll
      for (int q = 0; q < P; q++) {
        float sv[2] = {0.f, 0.f}, tv[2] = {0.f, 0.f}, zi[3] = {0.f, 0.f, 0.f};
        int u = 0;
#pragma unroll
        for (int c = 0; c < C; c++) {
          float zc = z[q][c];
          zi[c] = zc;
          if (!b[c]) {
            float s_ = p.tanh_out ? p.out_scale * tanh_sfu(so[q][c]) : so[q][c];
            float t_ = p.tanh_out ? p.out_scale * tanh_sfu(to[q][c]) : to[q][c];
            if (!isfinite(s_)) s_ = NAN;
            if (!isfinite(t_)) t_ = NAN;
            zc = fmaf(z[q][c], (p.tanh_out && p.out_scale == 1.f) ? exp_sfu(s_) : expf(s_), t_);
            if (u == 0) { sv[0] = s_; tv[0] = t_; } else { sv[1] = s_; tv[1] = t_; }
            u++;
          }
          z[q][c] = fmaf(zc, tail[2 * C + c], tail[3 * C + c]);      // ActNorm: z * exp(s) + t, exp(s) staged once per CTA
        }
        if (p.zin && ok[q]) {
          float4* rec = reinterpret_cast<float4*>(p.zin + (((int64_t)o * p.F + f) * p.N + n[q]) * RW);
          if (C == 2) rec[0] = make_float4(zi[0], zi[1], sv[0], tv[0]);
          else { rec[0] = make_float4(zi[0], zi[1], zi[2], sv[0]); rec[1] = make_float4(sv[1], tv[0], tv[1], 0.f); }
        }
      }
    }
#pragma unroll
    for (int q = 0; q < P; q++) {
      if (!ok[q]) continue;
      float xd[3] = {0.f, 0.f, 0.f};
#pragma unroll
      for (int c = 0; c < C; c++) xd[c] = mm_fwd(z[q][c], p.fc.new_min, p.fc.new_max, p.fc.nmin[c], p.fc.nmax[c]);
      *reinterpret_cast<float4*>(p.X + ((int64_t)o * p.N + n[q]) * 4) = make_float4(xd[0], xd[1], xd[2], 1.f);
      if (p.deformed) {
#pragma unroll
        for (int c = 0; c < C; c++) p.deformed[((int64_t)o * p.N + n[q]) * C + c] = xd[c];
      }
    }
    return true;
  };
  int64_t base = r0;
  bool more = true;
#pragma unroll 1
  for (int r = 0; r < p.rounds && more; r++, base += (int64_t)FLOW_P * T) more = round(std::integral_constant<int, FLOW_P>{}, base);
#pragma unroll 1
  for (int r = 0; r < p.rounds1 && more; r++, base += T) more = round(std::integral_constant<int, 1>{}, base);
}

// ---------------------------------------------------------------- inverse (PathConnectedNet.inverse, path_connected_net.py:107-122)
// x (a get_deformation output) -> MinMax -> flows in reverse order, each inverted (ActNorm: (z - t) exp(-s);
// coupling: zm + (1 - b)(z - t(zm)) exp(-s(zm)), normflows MaskedAffineFlow.inverse) -> inverse MinMax -> inverse 1x1 conv.
template <int C>
__global__ void __launch_bounds__(256) k_flow_inv(FlowP p, float* out) {
  extern __shared__ float sp[];   // [P_flow + 2C]
  const int o = blockIdx.y;
  const float* par = p.params + (int64_t)o * p.P + p.off_flow;
  const int PF = (int)p.P_flow + 2 * C;
  for (int i = threadIdx.x; i < PF; i += blockDim.x) sp[i] = par[i];
  __syncthreads();
  int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.N) return;
  const float* lin = sp + p.P_flow;
  float z[C];
#pragma unroll
  for (int c = 0; c < C; c++) z[c] = mm_fwd(coord(p.g, n, c), p.fc.nmin[c], p.fc.nmax[c], p.fc.new_min, p.fc.new_max);
  const int m = p.m;
  const int half = 2 * m * C + m + C;
  for (int f = p.F - 1; f >= 0; f--) {
    const float* w = sp + (int64_t)f * p.per_flow;
    const float* an = w + 2 * half;
    float zm[C];
    bool b[C];
#pragma unroll
    for (int c = 0; c < C; c++) {
      z[c] = (z[c] - an[C + c]) * expf(-an[c]);          // ActNorm inverse
      b[c] = p.fc.masks[f * C + c] != 0; zm[c] = b[c] ? z[c] : 0.f;
    }
    float so[C], to[C];
#pragma unroll
    for (int c = 0; c < C; c++) { so[c] = w[m * C + m + C * m + c]; to[c] = w[half + m * C + m + C * m + c]; }
    for (int k = 0; k < m; k++) {
      float ps = w[m * C + k], pt = w[half + m * C + k];
#pragma unroll
      for (int c = 0; c < C; c++) { ps = fmaf(w[k * C + c], zm[c], ps); pt = fmaf(w[half + k * C + c], zm[c], pt); }
      float hs = fmaxf(ps, 0.f), ht = fmaxf(pt, 0.f);
#pragma unroll
      for (int c = 0; c < C; c++) {
        so[c] = fmaf(w[m * C + m + c * m + k], hs, so[c]);
        to[c] = fmaf(w[half + m * C + m + c * m + k], ht, to[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < C; c++) {
      float s_ = p.tanh_out ? p.out_scale * tanhf(so[c]) : so[c];
      float t_ = p.tanh_out ? p.out_scale * tanhf(to[c]) : to[c];
      if (!isfinite(s_)) s_ = NAN;
      if (!isfinite(t_)) t_ = NAN;
      if (!b[c]) z[c] = (z[c] - t_) * expf(-s_);
    }
  }
#pragma unroll
  for (int c = 0; c < C; c++) {
    float x = mm_fwd(z[c], p.fc.new_min, p.fc.new_max, p.fc.nmin[c], p.fc.nmax[c]);
    out[((int64_t)o * p.N + n) * C + c] = (1.0f / lin[c]) * (x - lin[C + c]);
  }
}

// ---------------------------------------------------------------- backward
// ONE kernel, no per-pixel record through global memory.  A CTA owns a pixel range and walks the flows in reverse; the
// running coordinate gradient dz of its pixels stays in shared memory between flows.  For one flow, every thread
// visits its pixels (P at a time, sharing each weight record) and accumulates IN REGISTERS, per hidden unit k and net,
// the masked sums every weight gradient of that unit is linear in:
//     A[k][u]    = sum_px [pre_k > 0] * d_u            (d_u = gradient at the pre-activation output u of the net)
//     B[k][u][c] = sum_px [pre_k > 0] * d_u * z_c      (c = masked input components)
// because  d pre_k = [pre_k > 0] * sum_u d_u W2[u][k]  factors into a per-pixel and a per-unit part:
//     dW1[k][c] = sum_u W2[u][k] B[k][u][c],  db1[k] = sum_u W2[u][k] A[k][u],
//     dW2[u][k] = sum_px d_u relu(pre_k) = b1[k] A[k][u] + sum_c W1[k][c] B[k][u][c],
// and the gradient reaching the masked inputs is  dz_c += sum_u d_u * (sum_k [pre_k > 0] W2[u][k] W1[k][c])  with the
// products W2[u][k] W1[k][c] staged per unit.  Per (pixel, unit, net): one FMA per masked input, one compare and
// 2 NU NM + NU predicated adds -- 10 instructions for C = 2 against 24 in the two-kernel version, and the cross-pixel
// reduction happens once per flow and CTA (warp reduce-scatter + fixed-order combine), not per pixel.
// The unit range is processed in blocks of KB units (32 for C = 2: one pass; 16 for C = 3: two passes over the pixels,
// 128 accumulator registers either way).
// Everything held in registers is indexed by ROLE (i-th masked component, j-th transformed component), everything in
// memory by component; which component plays which role is a run-time property of the flow.  One instantiation per number
// of masked components NM therefore serves every mask pattern (C = 2: one body for both alternating masks -- the two
// specialised copies did not fit the instruction cache together).
template <int C, int NM> struct FlowBwdCfg {
  static constexpr int NU = C - NM;
  static constexpr int NA1 = NU * (1 + NM);        // accumulators per unit and net
  static constexpr int NACC = 2 * NA1;
  static constexpr int KB = C == 2 ? 32 : 16;
  static constexpr int NPASS = 32 / KB;
};
template <int C> struct FlowBwdPack {
  static constexpr int RKB = C == 2 ? 8 : 12;      // floats per unit: [w1s[NM] | b1s | vs[NU][NM] | w1t[NM] | b1t | vt[NU][NM]]
  __host__ __device__ static int flow_stride() { return 32 * RKB + 4; }   // + exp(ActNorm.s)[C], pad
};

template <int C>
__device__ void stage_flow_bwd(const float* __restrict__ par, int F, int m, int64_t per_flow, float* sp, const FlowConsts& fc) {
  constexpr int RKB = FlowBwdPack<C>::RKB;
  const int half = 2 * m * C + m + C, FS = FlowBwdPack<C>::flow_stride();
  for (int t = threadIdx.x; t < F * 32; t += blockDim.x) {
    const int f = t >> 5, k = t & 31;
    const float* w = par + (int64_t)f * per_flow;
    float* r = sp + f * FS + k * RKB;
    int mb = 0;
#pragma unroll
    for (int c = 0; c < C; c++) mb |= fc.masks[f * C + c] != 0 ? 1 << c : 0;
#pragma unroll
    for (int i = 0; i < RKB; i++) r[i] = 0.f;          // units k >= m: pre-activation 0 -> never active
    if (k >= m) continue;
    int pos = 0;
    for (int net = 0; net < 2; net++) {
      const float* wn = w + net * half;
      for (int c = 0; c < C; c++) if ((mb >> c) & 1) r[pos++] = wn[k * C + c];                   // W1[k][c], masked c
      r[pos++] = wn[m * C + k];                                                                  // b1[k]
      for (int u = 0; u < C; u++) if (!((mb >> u) & 1))
        for (int c = 0; c < C; c++) if ((mb >> c) & 1) r[pos++] = wn[m * C + m + u * m + k] * wn[k * C + c];   // W2[u][k] W1[k][c]
    }
  }
  for (int t = threadIdx.x; t < F * 4; t += blockDim.x) {
    const int f = t >> 2, c = t & 3;
    const float* w = par + (int64_t)f * per_flow;
    sp[f * FS + 32 * RKB + c] = c < C ? expf(w[2 * half + c]) : 0.f;
  }
}

__device__ __forceinline__ float gate_gt0(float x) {      // x > 0 ? 1.0f : 0.0f  (FSET.BF.GT)
  float g;
  asm("set.gt.f32.f32 %0, %1, 0f00000000;" : "=f"(g) : "f"(x));
  return g;
}

// Sum of v[i] over the 32 lanes for 32 values at once: afterwards lane l holds the total of value l (31 shuffles).
__device__ __forceinline__ float warp_reduce_scatter32(float* v, int lane) {
#pragma unroll
  for (int off = 16, n = 32; off >= 1; off >>= 1, n >>= 1) {
    const bool up = lane & off;
#pragma unroll
    for (int k = 0; k < 16; k++) {
      if (k < n / 2) {
        const float send = up ? v[k] : v[k + n / 2];
        const float keep = up ? v[k + n / 2] : v[k];
        v[k] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
  }
  return v[0];
}

template <int C> __device__ __forceinline__ float pick(const float* v, int c) {   // v[c] for a run-time c, v in registers
  return C == 2 ? (c == 0 ? v[0] : v[1]) : (c == 0 ? v[0] : (c == 1 ? v[1] : v[2]));
}

struct FlowBwdShared {
  float* wrec;     // staged weights (stage_flow_bwd)
  float* red;      // 2 x FLOW_RED_FLOATS: double-buffered reduction scratch
  float* stage;    // [2][P][T] saved records of the next round, filled by cp.async (per-thread slots)
  float* dzp;      // partial masked-input gradient between unit passes (C = 3): [C][chunk] in shared memory or [n][4] global
  int dzp_cs, dzp_ps;
};

// the full rounds of the backward walk in execution order: flows in reverse, unit passes, rounds
struct FlowStep {
  int f, pass, r;
  __device__ __forceinline__ bool valid() const { return f >= 0; }
  __device__ __forceinline__ void next(int npass, int rounds) {
    if (++r < rounds) return;
    r = 0;
    if (++pass < npass) return;
    pass = 0;
    --f;
  }
};

// cp.async of this thread's P records of one round into its private slots of a staging buffer
template <int C, int P>
__device__ __forceinline__ void prefetch_round(const FlowP& p, float* stage_buf, const FlowStep& st, int o, int64_t r0, int len) {
  constexpr int RW = FlowSave<C>::RW;
  const int T = blockDim.x, tid = threadIdx.x;
  const float* zrec = p.zin + ((((int64_t)o * p.F + st.f) * p.N) + r0) * RW;      // this CTA's range of the flow's records
  const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(stage_buf);
#pragma unroll
  for (int q = 0; q < P; q++) {
    const int loc = (st.r * P + q) * T + tid;                                     // 32-bit index inside the range
    if (loc < len) {
#pragma unroll
      for (int i = 0; i < RW / 4; i++)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sbase + (uint32_t)(((q * (RW / 4) + i) * T + tid) * 16)),
                     "l"(zrec + (uint32_t)(loc * RW + 4 * i)) : "memory");
    }
  }
}

// one flow with NM masked components (mask pattern mb) over the CTA's pixel range
template <int C, int NM>
__device__ __forceinline__ void flow_bwd_one(const FlowP& p, const FlowBwdShared& sh, int f, int mb, int o, int64_t r0, int64_t r1,
                                             float* dzg, int dz_cs, int dz_ps, FlowStep& pre, int& buf) {
  using Cf = FlowBwdCfg<C, NM>;
  constexpr int NU = Cf::NU, NA1 = Cf::NA1, NACC = Cf::NACC, KB = Cf::KB, NPASS = Cf::NPASS;
  constexpr int RKB = FlowBwdPack<C>::RKB, RW = FlowSave<C>::RW;
  const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = T >> 5;
  const int m = p.m, half = 2 * m * C + m + C;
  const float* wf = sh.wrec + f * FlowBwdPack<C>::flow_stride();
  const float* zrec = p.zin + (((int64_t)o * p.F + f) * p.N) * RW;
  // roles: mi[i] = i-th masked component, ui[j] = j-th transformed component (ascending)
  int mi[NM], ui[NU];
  {
    int a = 0, b = 0;
#pragma unroll
    for (int c = 0; c < C; c++) {
      if ((mb >> c) & 1) { if (a < NM) mi[a] = c; a++; } else { if (b < NU) ui[b] = c; b++; }
    }
  }
  float ea_m[NM], ea_u[NU];
#pragma unroll
  for (int i = 0; i < NM; i++) ea_m[i] = wf[32 * RKB + mi[i]];
#pragma unroll
  for (int j = 0; j < NU; j++) ea_u[j] = wf[32 * RKB + ui[j]];
  // per-thread scalar sums: d ActNorm.s / .t of the masked and of the transformed components, d s.b2 / d t.b2
  float sas_m[NM], sat_m[NM], sas_u[NU], sat_u[NU], sb2s[NU], sb2t[NU];
#pragma unroll
  for (int i = 0; i < NM; i++) { sas_m[i] = 0.f; sat_m[i] = 0.f; }
#pragma unroll
  for (int j = 0; j < NU; j++) { sas_u[j] = 0.f; sat_u[j] = 0.f; sb2s[j] = 0.f; sb2t[j] = 0.f; }

#pragma unroll 1
  for (int pass = 0; pass < NPASS; pass++) {
    float acc[KB * NACC];
#pragma unroll
    for (int i = 0; i < KB * NACC; i++) acc[i] = 0.f;
    const float* wk = wf + pass * KB * RKB;
    const bool last_pass = pass == NPASS - 1;
    // one round: P pixels of this thread starting at `base` (slot q -> pixel base + q * T + tid), all sharing the records;
    // src: this thread's staged records (full rounds) or null (remainder rounds read global memory)
    const int len = (int)(r1 - r0);
    const float* zrec_cta = zrec + r0 * RW;
    auto round = [&](auto p_c, int base, const float* src) -> bool {      // base: local index of the round's first pixel
      constexpr int P = decltype(p_c)::value;
      bool ok[P];
      float zm[P][NM], ds[P][NU], dt[P][NU], us[P][NU * NM], ut[P][NU * NM], Ds[P][NU * NM], Dt[P][NU * NM];
      float dzo_u[P][NU];
#pragma unroll
      for (int q = 0; q < P; q++) {
        const int n = base + q * T + tid;
        ok[q] = n < len;
        float z[3] = {0.f, 0.f, 0.f}, s[2] = {0.f, 0.f}, t[2] = {0.f, 0.f}, dz[3] = {0.f, 0.f, 0.f};
        if (ok[q]) {
          float4 a, b4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (src) {
            a = *reinterpret_cast<const float4*>(src + ((q * (RW / 4)) * T + tid) * 4);
            if (C == 3) b4 = *reinterpret_cast<const float4*>(src + ((q * (RW / 4) + (RW / 4 - 1)) * T + tid) * 4);
          } else {
            a = *reinterpret_cast<const float4*>(zrec_cta + (uint32_t)(n * RW));
            if (C == 3) b4 = *reinterpret_cast<const float4*>(zrec_cta + (uint32_t)(n * RW + 4));
          }
          if (C == 2) { z[0] = a.x; z[1] = a.y; s[0] = a.z; t[0] = a.w; }
          else { z[0] = a.x; z[1] = a.y; z[2] = a.z; s[0] = a.w; s[1] = b4.x; t[0] = b4.y; t[1] = b4.z; }
#pragma unroll
          for (int c = 0; c < C; c++) dz[c] = dzg[c * dz_cs + n * dz_ps];
        }
#pragma unroll
        for (int i = 0; i < NM; i++) {          // masked components pass through the coupling
          const float zc = pick<C>(z, mi[i]), dzc = pick<C>(dz, mi[i]);
          zm[q][i] = zc;
          if (last_pass) { sas_m[i] = fmaf(dzc * zc, ea_m[i], sas_m[i]); sat_m[i] += dzc; }
        }
#pragma unroll
        for (int j = 0; j < NU; j++) {          // transformed components: z' = z exp(s) + t
          const float zc = pick<C>(z, ui[j]), dzc = pick<C>(dz, ui[j]);
          const float dzp = dzc * ea_u[j];
          const float e = (p.tanh_out && p.out_scale == 1.f) ? exp_sfu(s[j]) : expf(s[j]);      // the same function as the forward
          const float isc = p.inv_out_scale;
          const float dsv = dzp * zc * e;
          ds[q][j] = p.tanh_out ? dsv * p.out_scale * (1.f - (s[j] * isc) * (s[j] * isc)) : dsv;     // d (c tanh a) / da = c (1 - tanh^2)
          dt[q][j] = p.tanh_out ? dzp * p.out_scale * (1.f - (t[j] * isc) * (t[j] * isc)) : dzp;
          dzo_u[q][j] = dzp * e;
          if (last_pass) {
            sas_u[j] = fmaf(dzc * fmaf(zc, e, t[j]), ea_u[j], sas_u[j]);
            sat_u[j] += dzc;
            sb2s[j] += ds[q][j];
            sb2t[j] += dt[q][j];
          }
#pragma unroll
          for (int i = 0; i < NM; i++) { us[q][j * NM + i] = ds[q][j] * zm[q][i]; ut[q][j * NM + i] = dt[q][j] * zm[q][i]; Ds[q][j * NM + i] = 0.f; Dt[q][j * NM + i] = 0.f; }
        }
      }
      if (!ok[0]) return false;       // slots are ordered: nothing left for this thread
      // ---- unit loop: all KB units of this pass, every record shared by the P pixels
#pragma unroll
      for (int k = 0; k < KB; k++) {
        float w[RKB];
#pragma unroll
        for (int i = 0; i < RKB / 4; i++) *reinterpret_cast<float4*>(&w[4 * i]) = reinterpret_cast<const float4*>(wk + k * RKB)[i];
        constexpr int OT = NM + 1 + NU * NM;       // offset of the t net inside the record
#pragma unroll
        for (int q = 0; q < P; q++) {
          float ps = w[NM], pt = w[OT + NM];
#pragma unroll
          for (int c = 0; c < NM; c++) { ps = fmaf(w[c], zm[q][c], ps); pt = fmaf(w[OT + c], zm[q][c], pt); }
          // gate = [pre > 0] as 1.0f / 0.0f (one FSET) and FMAs instead of predicated adds
          float* a = &acc[k * NACC];
          const float gs = gate_gt0(ps), gt = gate_gt0(pt);
#pragma unroll
          for (int u = 0; u < NU; u++) {
            a[u * (1 + NM)] = fmaf(gs, ds[q][u], a[u * (1 + NM)]);
            a[NA1 + u * (1 + NM)] = fmaf(gt, dt[q][u], a[NA1 + u * (1 + NM)]);
#pragma unroll
            for (int c = 0; c < NM; c++) {
              a[u * (1 + NM) + 1 + c] = fmaf(gs, us[q][u * NM + c], a[u * (1 + NM) + 1 + c]);
              Ds[q][u * NM + c] = fmaf(gs, w[NM + 1 + u * NM + c], Ds[q][u * NM + c]);
              a[NA1 + u * (1 + NM) + 1 + c] = fmaf(gt, ut[q][u * NM + c], a[NA1 + u * (1 + NM) + 1 + c]);
              Dt[q][u * NM + c] = fmaf(gt, w[OT + NM + 1 + u * NM + c], Dt[q][u * NM + c]);
            }
          }
        }
      }
      // ---- gradient reaching the inputs of this coupling
#pragma unroll
      for (int q = 0; q < P; q++) {
        if (!ok[q]) continue;
        const int n = base + q * T + tid;
#pragma unroll
        for (int i = 0; i < NM; i++) {
          float g = 0.f;
#pragma unroll
          for (int u = 0; u < NU; u++) g = fmaf(ds[q][u], Ds[q][u * NM + i], fmaf(dt[q][u], Dt[q][u * NM + i], g));
          if (NPASS > 1 && pass > 0) g += sh.dzp[mi[i] * sh.dzp_cs + n * sh.dzp_ps];
          if (!last_pass) sh.dzp[mi[i] * sh.dzp_cs + n * sh.dzp_ps] = g;
          else dzg[mi[i] * dz_cs + n * dz_ps] = fmaf(dzg[mi[i] * dz_cs + n * dz_ps], ea_m[i], g);      // dz * exp(ActNorm.s) + MLP path
        }
        if (last_pass) {
#pragma unroll
          for (int j = 0; j < NU; j++) dzg[ui[j] * dz_cs + n * dz_ps] = dzo_u[q][j];
        }
      }
      return true;
    };
    {
      int base = 0;
      bool more = true;
#pragma unroll 1
      for (int r = 0; r < p.rounds; r++, base += FLOW_PB * T) {
        // records of this round were requested one round ago; request the next full round (of whatever flow) now
        float* cur = sh.stage + buf * (FLOW_PB * (RW / 4) * T * 4);
        buf ^= 1;
        pre.next(NPASS, p.rounds);
        if (pre.valid()) prefetch_round<C, FLOW_PB>(p, sh.stage + buf * (FLOW_PB * (RW / 4) * T * 4), pre, o, r0, (int)(r1 - r0));
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        if (more) more = round(std::integral_constant<int, FLOW_PB>{}, base, cur);
      }
#pragma unroll 1
      for (int r = 0; r < p.rounds1 && more; r++, base += T) more = round(std::integral_constant<int, 1>{}, base, nullptr);
    }
    // ---- cross-pixel reduction of this pass's KB units: warp reduce-scatter into the warp's row of `red`, ONE block barrier,
    // then one thread per (net, unit) adds up the warps' rows in a fixed order and converts the sums into gradients.  The
    // scratch is double buffered over (flow, pass): the writes of the next reduction go to the other half, and the one after
    // that is separated from these reads by the next barrier -- no trailing barrier, the other warps run on into the next flow.
    float* red = sh.red + ((f * NPASS + pass) & 1) * FLOW_RED_FLOATS;      // [16 warps][128] | [16 warps][16]
    float* red2 = red + 16 * 128;
#pragma unroll
    for (int b = 0; b < KB * NACC / 32; b++) red[warp * 128 + b * 32 + lane] = warp_reduce_scatter32(&acc[b * 32], lane);
    if (last_pass) {
      // scalar sums of the flow: ActNorm pair and the output biases of s / t; red2 rows: [as(C) | at(C) | b2s(C) | b2t(C)]
      auto wsum = [&](float a) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
        return a;
      };
      if (lane < 16) red2[warp * 16 + lane] = 0.f;
      __syncwarp();
#pragma unroll
      for (int i = 0; i < NM; i++) {
        const float a = wsum(sas_m[i]), b2 = wsum(sat_m[i]);
        if (lane == 0) { red2[warp * 16 + mi[i]] = a; red2[warp * 16 + C + mi[i]] = b2; }
      }
#pragma unroll
      for (int j = 0; j < NU; j++) {
        const float a = wsum(sas_u[j]), b2 = wsum(sat_u[j]), c2 = wsum(sb2s[j]), d2 = wsum(sb2t[j]);
        if (lane == 0) { red2[warp * 16 + ui[j]] = a; red2[warp * 16 + C + ui[j]] = b2; red2[warp * 16 + 2 * C + ui[j]] = c2; red2[warp * 16 + 3 * C + ui[j]] = d2; }
      }
    }
    __syncthreads();
    // (pointers of the conversion are formed here, not at the top: nothing of them stays live across the unit loop)
    const float* wglob = p.params + (int64_t)o * p.P + p.off_flow + (int64_t)f * p.per_flow;
    float* out = p.fpart + ((int64_t)blockIdx.x * p.O + o) * (p.P_flow + 2 * C) + (int64_t)f * p.per_flow;
    for (int i = tid; i < 2 * KB; i += T) {
      const int net = i / KB, k = i - net * KB, kk = pass * KB + k;
      if (kk >= m) continue;
      const float* wn = wglob + net * half;
      float a[NA1];
#pragma unroll
      for (int x = 0; x < NA1; x++) {
        float t = 0.f;
        for (int w = 0; w < nwarps; w++) t += red[w * 128 + k * NACC + net * NA1 + x];
        a[x] = t;
      }
      float* on = out + net * half;
      float gb1 = 0.f, gw1[NM];
#pragma unroll
      for (int c = 0; c < NM; c++) gw1[c] = 0.f;
      const float b1 = wn[m * C + kk];
#pragma unroll
      for (int c = 0; c < C; c++) { on[kk * C + c] = 0.f; on[m * C + m + c * m + kk] = 0.f; }   // W1 columns of transformed inputs / W2 rows of masked outputs
#pragma unroll
      for (int u = 0; u < NU; u++) {
        const float w2 = wn[m * C + m + ui[u] * m + kk];
        gb1 = fmaf(w2, a[u * (1 + NM)], gb1);
        float gw2 = b1 * a[u * (1 + NM)];
#pragma unroll
        for (int c = 0; c < NM; c++) {
          gw1[c] = fmaf(w2, a[u * (1 + NM) + 1 + c], gw1[c]);
          gw2 = fmaf(wn[kk * C + mi[c]], a[u * (1 + NM) + 1 + c], gw2);
        }
        on[m * C + m + ui[u] * m + kk] = gw2;                                // d W2[u][k]
      }
#pragma unroll
      for (int c = 0; c < NM; c++) on[kk * C + mi[c]] = gw1[c];               // d W1[k][c]
      on[m * C + kk] = gb1;                                                  // d b1[k]
    }
    if (last_pass) {
      for (int x = (tid + T - (2 * KB) % T) % T; x < 4 * C; x += T) {      // threads next to the conversion ones (any block size)
        const int qd = x / C, c = x - qd * C;      // 0: ActNorm.s, 1: ActNorm.t, 2: s.b2, 3: t.b2
        float a = 0.f;
        for (int w = 0; w < nwarps; w++) a += red2[w * 16 + x];
        if (qd == 2) out[m * C + m + C * m + c] = a;
        else if (qd == 3) out[half + m * C + m + C * m + c] = a;
        else if (qd == 0) out[2 * half + c] = a;
        else out[2 * half + C + c] = a;
      }
    }
  }
}

// DG: also write the coordinate gradient p.dgrid (a separate instantiation, so that the fit path's code is untouched)
template <int C, bool DG>
__global__ void __launch_bounds__(FLOW_BWD_T, 1) k_flow_bwd(FlowP p) {
  extern __shared__ __align__(16) float sp[];
  constexpr int RW = FlowSave<C>::RW;
  const int o = blockIdx.y, tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = T >> 5;
  const float* par = p.params + (int64_t)o * p.P + p.off_flow;
  const int PF = (int)p.P_flow + 2 * C;
  const int64_t r0 = (int64_t)blockIdx.x * p.chunk, r1 = r0 + p.chunk < p.N ? r0 + p.chunk : p.N;
  FlowBwdShared sh;
  sh.wrec = sp;
  sh.red = sp + p.F * FlowBwdPack<C>::flow_stride();
  sh.stage = sh.red + 2 * FLOW_RED_FLOATS;
  float* after = sh.stage + 2 * FLOW_PB * (RW / 4) * FLOW_BWD_T * 4;
  float* dzs = p.dz_smem ? after : nullptr;
  sh.dzp = p.dz_smem ? after + C * p.chunk : p.dzp_g + ((int64_t)o * p.N + r0) * 4;   // C = 3 only (two unit passes)
  sh.dzp_cs = p.dz_smem ? (int)p.chunk : 1; sh.dzp_ps = p.dz_smem ? 1 : 4;
  stage_flow_bwd<C>(par, p.F, p.m, p.per_flow, sp, p.fc);
  float* outb = p.fpart + ((int64_t)blockIdx.x * p.O + o) * PF;
  if (r0 >= p.N) {          // empty range (rounded-up chunk): its partial is all zeros
    for (int i = tid; i < PF; i += T) outb[i] = 0.f;
    return;
  }
  // saved records of the first full round (last flow) are requested before anything else
  constexpr int NPASS = FlowBwdCfg<C, 1>::NPASS;
  FlowStep pre = {p.F - 1, 0, -1};
  int buf = 0;
  if (p.rounds > 0) {
    pre.r = 0;
    prefetch_round<C, FLOW_PB>(p, sh.stage, pre, o, r0, (int)(r1 - r0));
    asm volatile("cp.async.commit_group;" ::: "memory");
  } else {
    pre.f = -1;
  }
  (void)NPASS;
  // running gradient: shared memory [C][chunk], or in place in dX ([n][4]) when the range is too large
  float* dzg = p.dz_smem ? dzs : p.dX + ((int64_t)o * p.N + r0) * 4;
  const int dz_cs = p.dz_smem ? (int)p.chunk : 1, dz_ps = p.dz_smem ? 1 : 4;
  for (int64_t n = r0 + tid; n < r1; n += T) {
    const float4 dx = *reinterpret_cast<const float4*>(p.dX + ((int64_t)o * p.N + n) * 4);
    const float d3[3] = {dx.x, dx.y, dx.z};
#pragma unroll
    for (int c = 0; c < C; c++)
      dzg[c * dz_cs + (int)(n - r0) * dz_ps] = d3[c] * ((p.fc.nmax[c] - p.fc.nmin[c]) / (p.fc.new_max - p.fc.new_min));
  }
  __syncthreads();          // staged weights; the dz slots are thread-private: pixel n is always handled by thread (n - r0) % T
  for (int f = p.F - 1; f >= 0; f--) {
    int mb = 0;
#pragma unroll
    for (int c = 0; c < C; c++) mb |= p.fc.masks[f * C + c] != 0 ? 1 << c : 0;
    const int nm = __popc(mb);
    if (nm == 1) flow_bwd_one<C, 1>(p, sh, f, mb, o, r0, r1, dzg, dz_cs, dz_ps, pre, buf);
    if constexpr (C == 3) {
      if (nm == 2) flow_bwd_one<C, 2>(p, sh, f, mb, o, r0, r1, dzg, dz_cs, dz_ps, pre, buf);
    }
  }
  // ---- 1x1-conv gradients (path_connected_net.py:65,82): fixed-order block reduction
  float glw[C], glb[C];
#pragma unroll
  for (int c = 0; c < C; c++) { glw[c] = 0.f; glb[c] = 0.f; }
  if (p.use_linear) {
    for (int64_t n = r0 + tid; n < r1; n += T) {
#pragma unroll
      for (int c = 0; c < C; c++) {
        const float dxc = dzg[c * dz_cs + (int)(n - r0) * dz_ps] * ((p.fc.new_max - p.fc.new_min) / (p.fc.nmax[c] - p.fc.nmin[c]));
        glw[c] = fmaf(dxc, coord(p.g, n, c), glw[c]);     // linear.weight
        glb[c] += dxc;                                     // linear.bias
      }
    }
  }
  if constexpr (DG) {       // coordinate gradient: linear.weight[c] * dxc (groups = C: weight [C,1,1,1]), one store per pixel
    float lw[C];
#pragma unroll
    for (int c = 0; c < C; c++) lw[c] = par[p.P_flow + c];
    for (int64_t n = r0 + tid; n < r1; n += T) {
#pragma unroll
      for (int c = 0; c < C; c++) {
        const float dxc = dzg[c * dz_cs + (int)(n - r0) * dz_ps] * ((p.fc.new_max - p.fc.new_min) / (p.fc.nmax[c] - p.fc.nmin[c]));
        p.dgrid[planar_index(p.g, n, c)] = lw[c] * dxc;
      }
    }
  }
  __syncthreads();          // the last flow's conversion threads are done with the scratch
  float* red2 = sh.red + 16 * 128;
#pragma unroll
  for (int c = 0; c < C; c++) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      glw[c] += __shfl_xor_sync(0xffffffffu, glw[c], off);
      glb[c] += __shfl_xor_sync(0xffffffffu, glb[c], off);
    }
    if (lane == 0) { red2[warp * 16 + c] = glw[c]; red2[warp * 16 + C + c] = glb[c]; }
  }
  __syncthreads();
  if (tid < 2 * C) {
    float a = 0.f;
    for (int w = 0; w < nwarps; w++) a += red2[w * 16 + tid];
    outb[p.P_flow + tid] = p.use_linear ? a : 0.f;
  }
}

// ======================================================================= C = 2: segment tables
// With two coordinates every coupling masks exactly one of them, so both of its MLPs are functions of ONE scalar:
//     net(z) = b2 + sum_k W2[k] relu(W1[k] z + b1[k])
// is piecewise linear in z with (at most) m breakpoints beta_k = -b1[k] / W1[k].  k_flow_tables sorts the breakpoints of every
// (flow, net) once per forward and tabulates slope and intercept of each of the m + 1 segments (sums in double, a unit that
// is active nowhere contributes an exact 0); the per-pixel work is then a 6-step branch-free search and ONE FMA per net
// instead of m (compare, max, FMA) triples, and the backward pass replaces the 4 m masked sums per pixel by 4 additions
// into the pixel's segment of a thread-private histogram in shared memory:
//     H0[j] = sum_{px in segment j} g,   H1[j] = sum_{px in segment j} g z        (g = gradient at the net's output)
// from which the masked sums of unit k follow as the sum over the segments where the unit is active (a suffix of the sorted
// segments for W1[k] > 0, a prefix for W1[k] < 0) -- summed as such, never as a difference of totals: a unit without active
// pixels gets an exactly zero gradient, as in the reference (Adam / Adamax would amplify any rounding residue to a full
// step).  No atomics: fixed summation order, results independent of the launch geometry of other objects.
// Table of one (flow, net): beta[32] sorted ascending (+inf padding) | (slope, intercept)[33] | info[32]: per UNIT its rank
// among the breakpoints | type << 8 (0: active above its breakpoint, 1: active below), -1 for k >= m | 2 pad.
// Table of one FLOW (both nets), FLOW_TAB floats:
//   [0, 64)      gamma: the breakpoints of both nets merged and sorted ascending (+inf padding) -- ONE search serves both nets
//   [64, 324)    per merged segment J = 0 .. 64: (slope_s, slope_t, intercept_s, intercept_t)
//   [324, 389)   per merged segment: 4 j_s | (4 j_t) << 16 -- the segment of each net (number of ITS breakpoints below z)
//   [392, 456)   per unit (net 0: 32, net 1: 32): rank among its net's breakpoints | type << 8 (0: active above its breakpoint,
//                1: active below), -1 for k >= m
constexpr int FLOW_TAB = 456;
constexpr int FLOW_TAB_FWD = 324;       // what the forward stages
constexpr int FLOW_TAB_SEG = 64;        // offset of the per-segment coefficients
constexpr int FLOW_TAB_JJ = 324;
constexpr int FLOW_TAB_INFO = 392;
constexpr int FLOW_SEG_ROWS = 132;      // histogram rows: (net, segment 0..32, {g, g z})

__global__ void __launch_bounds__(64) k_flow_tables(FlowP p) {
  const unsigned full = 0xffffffffu;
  const int f = blockIdx.x, o = blockIdx.y, lane = threadIdx.x & 31, net = threadIdx.x >> 5;
  const int m = p.m, half = 4 * m + m + 2;
  const float* wn = p.params + (int64_t)o * p.P + p.off_flow + (int64_t)f * p.per_flow + net * half;
  const int cm = p.fc.masks[f * 2] != 0 ? 0 : 1, cu = 1 - cm;
  __shared__ float sb[2][32], sS[2][33], sI[2][33];
  __shared__ int rank_of[2][32], flag[64];
  float w = 0.f, b = 0.f, v = 0.f;
  if (lane < m) { w = wn[lane * 2 + cm]; b = wn[2 * m + lane]; v = wn[2 * m + m + cu * m + lane]; }
  const float c0 = wn[2 * m + m + 2 * m + cu];
  // breakpoint and type; W1 = 0: a constant unit (always active for b1 > 0: "below +inf"; never otherwise: "above +inf")
  float beta = INFINITY;
  int type = 0;
  if (w > 0.f) { beta = -b / w; }
  else if (w < 0.f) { beta = -b / w; type = 1; }
  else if (b > 0.f) { type = 1; }
  if (!(beta == beta)) beta = INFINITY;
  if (lane >= m) { type = 0; v = 0.f; }
  // bitonic sort of (beta, unit) across the warp (one warp per net)
  float kb = beta;
  int ki = lane;
#pragma unroll
  for (int k2 = 2; k2 <= 32; k2 <<= 1) {
#pragma unroll
    for (int j = k2 >> 1; j > 0; j >>= 1) {
      const float ob = __shfl_xor_sync(full, kb, j);
      const int oi = __shfl_xor_sync(full, ki, j);
      const bool asc = (lane & k2) == 0, lower = (lane & j) == 0;
      const bool other_less = ob < kb || (ob == kb && oi < ki);
      if ((lower == asc) ? other_less : !other_less) { kb = ob; ki = oi; }
    }
  }
  // lane r now holds the r-th smallest breakpoint of its net and the unit it belongs to
  const float ws_ = __shfl_sync(full, w, ki), bs_ = __shfl_sync(full, b, ki), vs_ = __shfl_sync(full, v, ki);
  const int ts_ = __shfl_sync(full, type, ki);
  const double a = (double)vs_ * (double)ws_, d = (double)vs_ * (double)bs_;
  double pa = ts_ == 0 ? a : 0.0, pd = ts_ == 0 ? d : 0.0;        // inclusive prefix over the "above" units
  double na = ts_ == 1 ? a : 0.0, nd = ts_ == 1 ? d : 0.0;        // inclusive suffix over the "below" units
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const double ua = __shfl_up_sync(full, pa, off), ud = __shfl_up_sync(full, pd, off);
    const double da = __shfl_down_sync(full, na, off), dd = __shfl_down_sync(full, nd, off);
    if (lane >= off) { pa += ua; pd += ud; }
    if (lane + off < 32) { na += da; nd += dd; }
  }
  // segment j of the net = number of its breakpoints below z: "above" units of rank < j and "below" units of rank >= j are active
  double ea = __shfl_up_sync(full, pa, 1), ed = __shfl_up_sync(full, pd, 1);
  if (lane == 0) { ea = 0.0; ed = 0.0; }
  sb[net][lane] = kb;
  sS[net][lane] = (float)(ea + na);
  sI[net][lane] = (float)((double)c0 + ed + nd);
  if (lane == 31) { sS[net][32] = (float)pa; sI[net][32] = (float)((double)c0 + pd); }
  rank_of[net][ki] = lane;
  __syncthreads();
  float* tab = p.tab + ((int64_t)o * p.F + f) * FLOW_TAB;
  reinterpret_cast<int*>(tab)[FLOW_TAB_INFO + net * 32 + lane] = lane < m ? (rank_of[net][lane] | (type << 8)) : -1;
  // merge: position of this breakpoint among all 64 (ties: net 0 first), then the segment of either net per merged segment
  int cnt = 0;
#pragma unroll 8
  for (int i = 0; i < 32; i++) cnt += net == 0 ? (sb[1][i] < kb ? 1 : 0) : (sb[0][i] <= kb ? 1 : 0);
  const int pos = lane + cnt;
  tab[pos] = kb;
  flag[pos] = net;
  __syncthreads();
  for (int J = threadIdx.x; J <= 64; J += 64) {
    int js = 0;
    for (int i = 0; i < J; i++) js += flag[i] == 0 ? 1 : 0;
    const int jt = J - js;
    *reinterpret_cast<float4*>(tab + FLOW_TAB_SEG + 4 * J) = make_float4(sS[0][js], sS[1][jt], sI[0][js], sI[1][jt]);
    reinterpret_cast<int*>(tab)[FLOW_TAB_JJ + J] = (4 * js) | ((4 * jt) << 16);
  }
}

// C = 3: the flows that mask ONE coordinate (three of the six mask patterns of net_factory.py:86-99) feed one scalar into
// their MLPs as well; each net has two outputs (the two transformed coordinates a < b).  Forward only -- the backward of
// C = 3 priors keeps the unit loops (its per-thread histogram would need 264 rows).  Table of one flow, FLOW_TAB3 floats:
//   [0, 64)     gamma, merged and sorted as for C = 2
//   [64, 584)   per merged segment J = 0 .. 64: (slope_sa, slope_sb, slope_ta, slope_tb, icpt_sa, icpt_sb, icpt_ta, icpt_tb)
// Flows with two masked coordinates leave their table untouched (never read).
__global__ void __launch_bounds__(64) k_flow_tables3(FlowP p) {
  const unsigned full = 0xffffffffu;
  const int f = blockIdx.x, o = blockIdx.y, lane = threadIdx.x & 31, net = threadIdx.x >> 5;
  int mb = 0;
#pragma unroll
  for (int c = 0; c < 3; c++) mb |= p.fc.masks[f * 3 + c] != 0 ? 1 << c : 0;
  if (__popc(mb) != 1) return;
  const int cm = __ffs(mb) - 1, ua = cm == 0 ? 1 : 0, ub = cm == 2 ? 1 : 2;
  const int m = p.m, half = 6 * m + m + 3;
  const float* wn = p.params + (int64_t)o * p.P + p.off_flow + (int64_t)f * p.per_flow + net * half;
  __shared__ float sb[2][32], sS[2][2][33], sI[2][2][33];
  __shared__ int flag[64];
  float w = 0.f, b = 0.f, va = 0.f, vb = 0.f;
  if (lane < m) { w = wn[lane * 3 + cm]; b = wn[3 * m + lane]; va = wn[3 * m + m + ua * m + lane]; vb = wn[3 * m + m + ub * m + lane]; }
  const float c0a = wn[3 * m + m + 3 * m + ua], c0b = wn[3 * m + m + 3 * m + ub];
  float beta = INFINITY;
  int type = 0;
  if (w > 0.f) { beta = -b / w; }
  else if (w < 0.f) { beta = -b / w; type = 1; }
  else if (b > 0.f) { type = 1; }
  if (!(beta == beta)) beta = INFINITY;
  if (lane >= m) { type = 0; va = 0.f; vb = 0.f; }
  float kb = beta;
  int ki = lane;
#pragma unroll
  for (int k2 = 2; k2 <= 32; k2 <<= 1) {
#pragma unroll
    for (int j = k2 >> 1; j > 0; j >>= 1) {
      const float ob = __shfl_xor_sync(full, kb, j);
      const int oi = __shfl_xor_sync(full, ki, j);
      const bool asc = (lane & k2) == 0, lower = (lane & j) == 0;
      const bool other_less = ob < kb || (ob == kb && oi < ki);
      if ((lower == asc) ? other_less : !other_less) { kb = ob; ki = oi; }
    }
  }
  const float ws_ = __shfl_sync(full, w, ki), bs_ = __shfl_sync(full, b, ki);
  const float vas = __shfl_sync(full, va, ki), vbs = __shfl_sync(full, vb, ki);
  const int ts_ = __shfl_sync(full, type, ki);
#pragma unroll
  for (int u = 0; u < 2; u++) {
    const double v = u == 0 ? (double)vas : (double)vbs;
    const double a = v * (double)ws_, d = v * (double)bs_;
    double pa = ts_ == 0 ? a : 0.0, pd = ts_ == 0 ? d : 0.0, na = ts_ == 1 ? a : 0.0, nd = ts_ == 1 ? d : 0.0;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const double xa = __shfl_up_sync(full, pa, off), xd = __shfl_up_sync(full, pd, off);
      const double ya = __shfl_down_sync(full, na, off), yd = __shfl_down_sync(full, nd, off);
      if (lane >= off) { pa += xa; pd += xd; }
      if (lane + off < 32) { na += ya; nd += yd; }
    }
    double ea = __shfl_up_sync(full, pa, 1), ed = __shfl_up_sync(full, pd, 1);
    if (lane == 0) { ea = 0.0; ed = 0.0; }
    const double c0 = u == 0 ? (double)c0a : (double)c0b;
    sS[net][u][lane] = (float)(ea + na);
    sI[net][u][lane] = (float)(c0 + ed + nd);
    if (lane == 31) { sS[net][u][32] = (float)pa; sI[net][u][32] = (float)(c0 + pd); }
  }
  sb[net][lane] = kb;
  __syncthreads();
  float* tab = p.tab + ((int64_t)o * p.F + f) * FLOW_TAB3;
  int cnt = 0;
#pragma unroll 8
  for (int i = 0; i < 32; i++) cnt += net == 0 ? (sb[1][i] < kb ? 1 : 0) : (sb[0][i] <= kb ? 1 : 0);
  const int pos = lane + cnt;
  tab[pos] = kb;
  flag[pos] = net;
  __syncthreads();
  for (int J = threadIdx.x; J <= 64; J += 64) {
    int js = 0;
    for (int i = 0; i < J; i++) js += flag[i] == 0 ? 1 : 0;
    const int jt = J - js;
    float4* e = reinterpret_cast<float4*>(tab + 64 + 8 * J);
    e[0] = make_float4(sS[0][0][js], sS[0][1][js], sS[1][0][jt], sS[1][1][jt]);
    e[1] = make_float4(sI[0][0][js], sI[0][1][js], sI[1][0][jt], sI[1][1][jt]);
  }
}

// tanh / exp of the segment kernels: ex2.approx.ftz / rcp.approx.ftz without the denormal fix-ups of __expf / __fdividef
// (5 + 2 instructions; tanh(0) = 0 exactly, saturates to +-1, NaN propagates; forward and backward use the same two)
__device__ __forceinline__ float ex2_ftz(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_ftz(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float tanh_seg(float a) { return fmaf(-2.f, rcp_ftz(ex2_ftz(a * 2.885390081777927f) + 1.f), 1.f); }
__device__ __forceinline__ float exp_seg(float s) { return ex2_ftz(s * 1.4426950408889634f); }

// forward: k_flow_fwd<2> with the two MLP loops replaced by the table lookups; same launch geometry, same saved records
__global__ void __launch_bounds__(256) k_flow_fwd_seg(FlowP p) {
  extern __shared__ __align__(16) float sp[];   // [F][FLOW_TAB_FWD] tables | [F][4] exp(an_s)[2], an_t[2] | [4] linear
  grid_dep_launch();      // plain launch (nothing to wait for); the next kernel's own griddepcontrol.wait orders it after this one
  const int o = blockIdx.y, T = blockDim.x;
  const float* par = p.params + (int64_t)o * p.P + p.off_flow;
  const int m = p.m, half = 4 * m + m + 2;
  {
    const float* tg = p.tab + (int64_t)o * p.F * FLOW_TAB;
    for (int i = threadIdx.x; i < p.F * (FLOW_TAB_FWD / 4); i += T) {
      const int fn = i / (FLOW_TAB_FWD / 4), j = i - fn * (FLOW_TAB_FWD / 4);
      reinterpret_cast<float4*>(sp)[i] = reinterpret_cast<const float4*>(tg + fn * FLOW_TAB)[j];
    }
    float* an = sp + p.F * FLOW_TAB_FWD;
    for (int i = threadIdx.x; i < p.F * 4; i += T) {
      const int f = i >> 2, q = i & 3;
      const float v = par[(int64_t)f * p.per_flow + 2 * half + q];
      an[i] = q < 2 ? expf(v) : v;
    }
    if (threadIdx.x < 4) an[p.F * 4 + threadIdx.x] = par[p.P_flow + threadIdx.x];
  }
  __syncthreads();
  const float* ans = sp + p.F * FLOW_TAB_FWD;
  const float* lin = ans + p.F * 4;
  const int64_t r0 = (int64_t)blockIdx.x * p.chunk, r1 = r0 + p.chunk < p.N ? r0 + p.chunk : p.N;
  const bool save = p.zin != nullptr;
  auto round = [&](auto p_c, int64_t base) -> bool {
    constexpr int P = decltype(p_c)::value;
    int64_t n[P];
    bool ok[P];
    float z0[P], z1[P];
    float4* rec[P];
#pragma unroll
    for (int q = 0; q < P; q++) {
      const int64_t nq = base + (int64_t)q * T + threadIdx.x;
      ok[q] = nq < r1;
      n[q] = ok[q] ? nq : (r1 > 0 ? r1 - 1 : 0);
      float x0 = coord(p.g, n[q], 0), x1 = coord(p.g, n[q], 1);
      if (p.use_linear) { x0 = x0 * lin[0] + lin[2]; x1 = x1 * lin[1] + lin[3]; }
      z0[q] = mm_fwd(x0, p.fc.nmin[0], p.fc.nmax[0], p.fc.new_min, p.fc.new_max);
      z1[q] = mm_fwd(x1, p.fc.nmin[1], p.fc.nmax[1], p.fc.new_min, p.fc.new_max);
      rec[q] = reinterpret_cast<float4*>(p.zin) + ((int64_t)o * p.F * p.N + n[q]);
    }
    if (!ok[0]) return false;
    // one coupling + ActNorm for the P pixels; zm: the masked coordinate (feeds the MLPs, passes through), zu: the transformed one
    auto couple = [&](uint32_t tb, float* zm, float* zu, float am, float bm, float au, float bu, bool m_first) {
      uint32_t J4[P];
      seg_find4_multi<P>(tb, zm, J4);
      float4 cf[P];
#pragma unroll
      for (int q = 0; q < P; q++) cf[q] = lds_f32x4(tb + FLOW_TAB_SEG * 4 + 4 * J4[q]);      // (slope_s, slope_t, intercept_s, intercept_t)
#pragma unroll
      for (int q = 0; q < P; q++) {
        const float s_ = tanh_seg(fmaf(cf[q].x, zm[q], cf[q].z)), t_ = tanh_seg(fmaf(cf[q].y, zm[q], cf[q].w));      // finite or NaN
        if (save && ok[q]) *rec[q] = m_first ? make_float4(zm[q], zu[q], s_, t_) : make_float4(zu[q], zm[q], s_, t_);
        zu[q] = fmaf(fmaf(zu[q], exp_seg(s_), t_), au, bu);
        zm[q] = fmaf(zm[q], am, bm);
      }
    };
#pragma unroll 1
    for (int f = 0; f < p.F; f++) {
      const uint32_t tb = (uint32_t)__cvta_generic_to_shared(sp + f * FLOW_TAB_FWD);
      const float4 an = *reinterpret_cast<const float4*>(ans + f * 4);      // exp(s0), exp(s1), t0, t1
      if (p.fc.masks[f * 2] != 0) couple(tb, z0, z1, an.x, an.z, an.y, an.w, true);          // component 0 is the masked one
      else couple(tb, z1, z0, an.y, an.w, an.x, an.z, false);
#pragma unroll
      for (int q = 0; q < P; q++) rec[q] += p.N;
    }
#pragma unroll
    for (int q = 0; q < P; q++) {
      if (!ok[q]) continue;
      const float xa = mm_fwd(z0[q], p.fc.new_min, p.fc.new_max, p.fc.nmin[0], p.fc.nmax[0]);
      const float xb = mm_fwd(z1[q], p.fc.new_min, p.fc.new_max, p.fc.nmin[1], p.fc.nmax[1]);
      *reinterpret_cast<float4*>(p.X + ((int64_t)o * p.N + n[q]) * 4) = make_float4(xa, xb, 0.f, 1.f);
      if (p.deformed) { p.deformed[((int64_t)o * p.N + n[q]) * 2] = xa; p.deformed[((int64_t)o * p.N + n[q]) * 2 + 1] = xb; }
    }
    return true;
  };
  int64_t base = r0;
  bool more = true;
#pragma unroll 1
  for (int r = 0; r < p.rounds && more; r++, base += (int64_t)FLOW_P * T) more = round(std::integral_constant<int, FLOW_P>{}, base);
#pragma unroll 1
  for (int r = 0; r < p.rounds1 && more; r++, base += T) more = round(std::integral_constant<int, 1>{}, base);
}

// Sum over the 32 lanes of N values at once (N = 32, 16, ...): afterwards every lane holds the total of value
// (lane >> log2(32 / N)); N - 1 + log2(32 / N) shuffles.
template <int N>
__device__ __forceinline__ float warp_reduce_scatter(float* v, int lane) {
  int off = 16;
#pragma unroll
  for (int n = N; n > 1; n >>= 1, off >>= 1) {
    const bool up = lane & off;
#pragma unroll
    for (int k = 0; k < N / 2; k++) {
      if (k < n / 2) {
        const float send = up ? v[k] : v[k + n / 2];
        const float keep = up ? v[k + n / 2] : v[k];
        v[k] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
  }
#pragma unroll
  for (; off >= 1; off >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], off);
  return v[0];
}

// backward: like k_flow_bwd<2> a CTA owns a pixel range, keeps the running gradient in shared memory, walks the flows in
// reverse and prefetches the saved records one round ahead with cp.async -- but the unit loop is the segment histogram, and
// the warps never meet inside the flow loop: histogram columns, gradient slots and staged records are thread-private, every
// warp sums ITS 32 columns after each flow (warp reduce-scatter, 32 rows at a time) and parks the 138 sums in an L2-resident
// scratch.  One block barrier after the last flow, then the warps' sums are added in a fixed order and converted into the
// gradients of all flows at once.
// Shared memory: tables [F][FLOW_TAB] | exp(an_s) [F][4] | 64 floats | staged records [2][P][T][4] | histogram [132][T]
// (afterwards: summed rows [F][FLOW_SEG_RS]) | running gradient [2][chunk] (DZS)
constexpr int FLOW_SEG_RS = 144;      // scratch floats per (flow, warp): 132 histogram rows | 6 scalar sums | pad
template <bool DZS, bool DG>
__global__ void __launch_bounds__(FLOW_BWD_T, 1) k_flow_bwd_seg(FlowP p) {
  extern __shared__ __align__(16) float sp[];
  constexpr int C = 2, RW = 4, P = FLOW_PB, T = FLOW_BWD_T;      // always 256 threads: strides are immediates
  constexpr int nwarps = T / 32;
  const unsigned full = 0xffffffffu;
  const int o = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* par = p.params + (int64_t)o * p.P + p.off_flow;
  const int PF = (int)p.P_flow + 2 * C;
  const int m = p.m, half = 4 * m + m + 2;
  const int64_t r0 = (int64_t)blockIdx.x * p.chunk, r1 = r0 + p.chunk < p.N ? r0 + p.chunk : p.N;
  float* tabs = sp;
  float* eas = tabs + p.F * FLOW_TAB;
  float* red2 = eas + p.F * 4;
  float* stage = red2 + 64;
  float* hist = stage + 2 * P * T * 4;
  float* dzs = hist + FLOW_SEG_ROWS * T;
  {
    // launched with programmatic stream serialization behind the fused ICNN kernel: everything here depends on kernels
    // further back in the stream only (the tables and the parameters of this step), dX is read after the wait
#pragma unroll 4
    for (int i = 0; i < FLOW_SEG_ROWS; i++) hist[i * T + tid] = 0.f;
    const float* tg = p.tab + (int64_t)o * p.F * FLOW_TAB;
    for (int i = tid; i < p.F * (FLOW_TAB / 4); i += T) reinterpret_cast<float4*>(tabs)[i] = reinterpret_cast<const float4*>(tg)[i];
    for (int i = tid; i < p.F * 4; i += T) {
      const int f = i >> 2, c = i & 3;
      eas[i] = c < C ? expf(par[(int64_t)f * p.per_flow + 2 * half + c]) : 0.f;
    }
  }
  grid_dep_wait();
  grid_dep_launch();
  float* outb = p.fpart + ((int64_t)blockIdx.x * p.O + o) * PF;
  if (r0 >= p.N) {
    for (int i = tid; i < PF; i += T) outb[i] = 0.f;
    return;
  }
  const int len = (int)(r1 - r0);
  // Every warp owns a CONTIGUOUS block of the range (slot i of a lane = pixel wbase + 32 i + lane): its pixels are
  // neighbours in the image, so they fall into few segments and the per-flow reduction below touches few rows.
  const int wl_full = (len + nwarps - 1) / nwarps;
  const int wbase = warp * wl_full;
  const int wlen = len - wbase < wl_full ? (len - wbase > 0 ? len - wbase : 0) : wl_full;
  const int n_rounds = p.rounds;
  auto prefetch = [&](float* stage_buf, int f, int r) {
    const float* zrec = p.zin + ((((int64_t)o * p.F + f) * p.N) + r0 + wbase) * RW;
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(stage_buf);
#pragma unroll
    for (int q = 0; q < P; q++) {
      const int li = (r * P + q) * 32 + lane;
      if (li < wlen)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sbase + (uint32_t)((q * T + tid) * 16)), "l"(zrec + (uint32_t)(li * RW)) : "memory");
    }
  };
  int pre_f = p.F - 1, pre_r = 0, buf = 0;
  if (n_rounds > 0) prefetch(stage, pre_f, 0);
  asm volatile("cp.async.commit_group;" ::: "memory");
  // running gradient: shared memory [2][chunk], or in place in dX ([n][4]) when the range is too large
  float* dzg = DZS ? dzs : p.dX + ((int64_t)o * p.N + r0) * 4;
  const int dz_cs = DZS ? (int)p.chunk : 1;
  constexpr int dz_ps = DZS ? 1 : 4;
  for (int n = tid; n < len; n += T) {
    const float4 dx = *reinterpret_cast<const float4*>(p.dX + ((int64_t)o * p.N + r0 + n) * 4);
    dzg[n * dz_ps] = dx.x * ((p.fc.nmax[0] - p.fc.nmin[0]) / (p.fc.new_max - p.fc.new_min));
    dzg[dz_cs + n * dz_ps] = dx.y * ((p.fc.nmax[1] - p.fc.nmin[1]) / (p.fc.new_max - p.fc.new_min));
  }
  __syncthreads();          // tables, initial gradient; from here on gradient slots, histogram columns and staged records are thread-private
  float* hmine = hist + tid;
  float* scr_w = p.segscr + ((((int64_t)blockIdx.x * p.O + o) * p.F) * 8 + warp) * FLOW_SEG_RS;
#pragma unroll 1
  for (int f = p.F - 1; f >= 0; f--) {
    const bool m0 = p.fc.masks[f * 2] != 0;
    const int cmi = m0 ? 0 : 1, cui = 1 - cmi;
    const uint32_t tb = (uint32_t)__cvta_generic_to_shared(tabs + f * FLOW_TAB);
    const float ea_m = eas[f * 4 + cmi], ea_u = eas[f * 4 + cui];
    float* dzm_p = dzg + cmi * dz_cs + wbase * dz_ps;
    float* dzu_p = dzg + cui * dz_cs + wbase * dz_ps;
    float sas_m = 0.f, sat_m = 0.f, sas_u = 0.f, sat_u = 0.f, sb2s = 0.f, sb2t = 0.f;
    uint32_t lo_s = 0xffffu, hi_s = 0u, lo_t = 0xffffu, hi_t = 0u;      // touched segments (x 4), per net
    const float* zrec_w = p.zin + ((((int64_t)o * p.F + f) * p.N) + r0 + wbase) * RW;
    // one round: slots i0 .. i0 + PP - 1 of this lane.  Branch-free (the PP pixels interleave): a slot past the warp's block
    // computes on zeros and stores nothing.
    // records of the first remainder slot: requested now, consumed after the full rounds
    const int li_rem = n_rounds * P * 32 + lane;
    float4 rec_rem = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.rounds1 > 0 && li_rem < wlen) rec_rem = __ldcg(reinterpret_cast<const float4*>(zrec_w + (uint32_t)(li_rem * RW)));
    auto round = [&](auto p_c, auto all_c, int i0, const float* src, const float4* reg) {
      constexpr int PP = decltype(p_c)::value;
      constexpr bool ALL = decltype(all_c)::value;      // every slot of the round holds a pixel for every lane: no predicates
      // breadth first over the PP pixels of the round (loads, then every step of the search for all of them, ...): their
      // dependent chains overlap
      bool ok[PP];
      int li[PP];
      float zm[PP], zu[PP], sv[PP], tv[PP], dzm[PP], dzu[PP];
#pragma unroll
      for (int q = 0; q < PP; q++) {
        li[q] = (i0 + q) * 32 + lane;
        ok[q] = ALL || li[q] < wlen;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        dzm[q] = 0.f; dzu[q] = 0.f;
        if (reg) a = *reg;
        else if (src) { if (ok[q]) a = *reinterpret_cast<const float4*>(src + (q * T + tid) * 4); }
        else if (ok[q]) a = *reinterpret_cast<const float4*>(zrec_w + (uint32_t)(li[q] * RW));
        if (ok[q]) { dzm[q] = dzm_p[li[q] * dz_ps]; dzu[q] = dzu_p[li[q] * dz_ps]; }
        zm[q] = m0 ? a.x : a.y; zu[q] = m0 ? a.y : a.x; sv[q] = a.z; tv[q] = a.w;
      }
      uint32_t J4[PP], js[PP], jt[PP];
      seg_find4_multi<PP>(tb, zm, J4);                                                  // merged segment (x 4)
      float2 sl[PP];
#pragma unroll
      for (int q = 0; q < PP; q++) {
        sl[q] = lds_f32x2(tb + FLOW_TAB_SEG * 4 + 4 * J4[q]);                           // slopes of the segment, both nets
        const uint32_t jj = lds_u32(tb + FLOW_TAB_JJ * 4 + J4[q]);                      // 4 j_s | 4 j_t << 16
        js[q] = jj & 0xffffu; jt[q] = jj >> 16;
      }
      float gs[PP], gt[PP];
#pragma unroll
      for (int q = 0; q < PP; q++) {
        const float dzp = dzu[q] * ea_u;
        const float e = exp_seg(sv[q]);                  // s = tanh(.), the same function as the forward
        const float dsv = dzp * zu[q] * e;
        gs[q] = dsv * (1.f - sv[q] * sv[q]);             // d tanh(a) / da = 1 - tanh^2
        gt[q] = dzp * (1.f - tv[q] * tv[q]);
        sas_m = fmaf(dzm[q] * zm[q], ea_m, sas_m); sat_m += dzm[q];
        sas_u = fmaf(dzu[q] * fmaf(zu[q], e, tv[q]), ea_u, sas_u); sat_u += dzu[q];
        sb2s += gs[q]; sb2t += gt[q];
        if (ok[q]) {
          dzm_p[li[q] * dz_ps] = fmaf(dzm[q], ea_m, fmaf(gs[q], sl[q].x, gt[q] * sl[q].y));
          dzu_p[li[q] * dz_ps] = dzp * e;
          lo_s = min(lo_s, js[q]); hi_s = max(hi_s, js[q]); lo_t = min(lo_t, jt[q]); hi_t = max(hi_t, jt[q]);
        }
      }
#pragma unroll
      for (int q = 0; q < PP; q++) {
        float* hs = hmine + (js[q] >> 1) * T;                  // rows 2 j, 2 j + 1
        float* ht = hmine + (66 + (jt[q] >> 1)) * T;
        if (ok[q]) {
          hs[0] += gs[q];
          hs[T] = fmaf(gs[q], zm[q], hs[T]);
          ht[0] += gt[q];
          ht[T] = fmaf(gt[q], zm[q], ht[T]);
        }
      }
    };
#pragma unroll 1
    for (int r = 0; r < n_rounds; r++) {
      // records of this round were requested one round ago; request the next full round (of whatever flow) now
      float* cur = stage + buf * (P * T * 4);
      buf ^= 1;
      if (++pre_r == n_rounds) { pre_r = 0; --pre_f; }
      if (pre_f >= 0) prefetch(stage + buf * (P * T * 4), pre_f, pre_r);
      asm volatile("cp.async.commit_group;" ::: "memory");
      asm volatile("cp.async.wait_group 1;" ::: "memory");
      if ((r * P + P) * 32 <= wlen) round(std::integral_constant<int, P>{}, std::true_type{}, r * P, cur, nullptr);
      else round(std::integral_constant<int, P>{}, std::false_type{}, r * P, cur, nullptr);
    }
    if (p.rounds1 > 0) round(std::integral_constant<int, 1>{}, std::false_type{}, n_rounds * P, nullptr, &rec_rem);
#pragma unroll 1
    for (int r = 1; r < p.rounds1; r++) round(std::integral_constant<int, 1>{}, std::false_type{}, n_rounds * P + r, nullptr, nullptr);
    // ---- this warp's 32 histogram columns -> row sums + 6 scalar sums in the scratch.  Only the segments some lane of the
    // warp touched in this flow (a contiguous range per net) are summed and zeroed again, four segments = 8 rows per
    // reduce-scatter; everything else is written as 0.  Fixed order (lane tree), no other warp involved.
    float* scr = scr_w + (int64_t)f * 8 * FLOW_SEG_RS;
#pragma unroll
    for (int i = 0; i < FLOW_SEG_RS; i += 32) if (i + lane < FLOW_SEG_RS) scr[i + lane] = 0.f;
    __syncwarp();
    {
      float v[8] = {sas_m, sat_m, sas_u, sat_u, sb2s, sb2t, 0.f, 0.f};
      const float a = warp_reduce_scatter<8>(v, lane);
      if ((lane & 3) == 0 && lane < 24) scr[132 + (lane >> 2)] = a;
    }
#pragma unroll 1
    for (int net = 0; net < 2; net++) {
      const int lo = (int)(__reduce_min_sync(full, net ? lo_t : lo_s) >> 2), hi = (int)(__reduce_max_sync(full, net ? hi_t : hi_s) >> 2);
#pragma unroll 1
      for (int j = lo & ~3; j <= hi; j += 4) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const int row = 2 * j + i;          // within the net: rows 0 .. 65
          v[i] = 0.f;
          if (row < 66) { v[i] = hmine[(net * 66 + row) * T]; hmine[(net * 66 + row) * T] = 0.f; }
        }
        const float a = warp_reduce_scatter<8>(v, lane);
        const int row = 2 * j + (lane >> 2);
        if ((lane & 3) == 0 && row < 66) scr[net * 66 + row] = a;
      }
    }
  }
  __syncthreads();          // every warp's gradient slots and scratch rows are written; the histogram is dead
  // ---- 1x1-conv gradients: fixed-order block reduction
  float glw[C] = {0.f, 0.f}, glb[C] = {0.f, 0.f};
  if (p.use_linear) {
    for (int n = tid; n < len; n += T) {
#pragma unroll
      for (int c = 0; c < C; c++) {
        const float dxc = dzg[c * dz_cs + n * dz_ps] * ((p.fc.new_max - p.fc.new_min) / (p.fc.nmax[c] - p.fc.nmin[c]));
        glw[c] = fmaf(dxc, coord(p.g, r0 + n, c), glw[c]);
        glb[c] += dxc;
      }
    }
  }
  if constexpr (DG) {       // coordinate gradient: linear.weight[c] * dxc, one store per pixel and channel
    const float lw0 = par[p.P_flow], lw1 = par[p.P_flow + 1];
    for (int n = tid; n < len; n += T) {
      p.dgrid[planar_index(p.g, r0 + n, 0)] = lw0 * (dzg[n * dz_ps] * ((p.fc.new_max - p.fc.new_min) / (p.fc.nmax[0] - p.fc.nmin[0])));
      p.dgrid[planar_index(p.g, r0 + n, 1)] =
          lw1 * (dzg[dz_cs + n * dz_ps] * ((p.fc.new_max - p.fc.new_min) / (p.fc.nmax[1] - p.fc.nmin[1])));
    }
  }
#pragma unroll
  for (int c = 0; c < C; c++) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      glw[c] += __shfl_xor_sync(full, glw[c], off);
      glb[c] += __shfl_xor_sync(full, glb[c], off);
    }
    if (lane == 0) { red2[warp * 4 + c] = glw[c]; red2[warp * 4 + C + c] = glb[c]; }
  }
  // ---- rows of all flows: the warps' sums in ascending warp order (read from L2)
  float* Hs = hist;
  {
    const float* scr_cta = p.segscr + (((int64_t)blockIdx.x * p.O + o) * p.F) * 8 * FLOW_SEG_RS;
    const int items = p.F * FLOW_SEG_RS;
#pragma unroll 2
    for (int i = tid; i < items; i += T) {
      const int f = i / FLOW_SEG_RS, row = i - f * FLOW_SEG_RS;
      const float* src = scr_cta + (int64_t)f * 8 * FLOW_SEG_RS + row;
      float v[nwarps];
#pragma unroll
      for (int w = 0; w < nwarps; w++) v[w] = __ldcg(src + w * FLOW_SEG_RS);
      float a = v[0];
#pragma unroll
      for (int w = 1; w < nwarps; w++) a += v[w];
      Hs[i] = a;
    }
  }
  __syncthreads();
  if (tid < 2 * C) {
    float a = 0.f;
    for (int w = 0; w < nwarps; w++) a += red2[w * 4 + tid];
    outb[p.P_flow + tid] = p.use_linear ? a : 0.f;
  }
  // ---- masked sums of every hidden unit = sum over the segments where it is active (a prefix or a suffix of the sorted
  // segments: warp scans, lane = segment, then lane = unit picks the entry of its rank), then the gradients.  A warp per
  // (flow, net).
#pragma unroll 1
  for (int pr = warp; pr < p.F * 2; pr += nwarps) {
    const int f = pr >> 1, net = pr & 1;
    const int cmi = p.fc.masks[f * 2] != 0 ? 0 : 1, cui = 1 - cmi;
    const float* hr = Hs + f * FLOW_SEG_RS + net * 66;
    const float* wn = par + (int64_t)f * p.per_flow + net * half;
    float* on = outb + (int64_t)f * p.per_flow + net * half;
    const int k = lane;
    float w1 = 0.f, b1 = 0.f, w2 = 0.f;
    int info = -1;
    if (k < m) {
      w1 = wn[k * 2 + cmi]; b1 = wn[2 * m + k]; w2 = wn[2 * m + m + cui * m + k];
      info = reinterpret_cast<const int*>(tabs + f * FLOW_TAB)[FLOW_TAB_INFO + net * 32 + k];
    }
    const float2 h = *reinterpret_cast<const float2*>(hr + 2 * lane);          // segment `lane`
    const float2 e = *reinterpret_cast<const float2*>(hr + 64);                // segment 32
    float p0 = h.x, p1 = h.y, s0 = h.x, s1 = h.y;      // inclusive prefix / suffix over segments 0 .. 31
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const float u0 = __shfl_up_sync(full, p0, off), u1 = __shfl_up_sync(full, p1, off);
      const float d0 = __shfl_down_sync(full, s0, off), d1 = __shfl_down_sync(full, s1, off);
      if (lane >= off) { p0 += u0; p1 += u1; }
      if (lane + off < 32) { s0 += d0; s1 += d1; }
    }
    s0 += e.x; s1 += e.y;                                // ... and segment 32
    const int rank = info & 0xff, type = info >> 8;
    // "above" units (type 0) are active in the segments rank + 1 .. 32, "below" units in 0 .. rank
    const int srcl = type == 0 ? (rank < 31 ? rank + 1 : 31) : rank;
    const float fs0 = __shfl_sync(full, s0, srcl & 31), fs1 = __shfl_sync(full, s1, srcl & 31);
    const float fp0 = __shfl_sync(full, p0, srcl & 31), fp1 = __shfl_sync(full, p1, srcl & 31);
    float a0 = type == 0 ? (rank < 31 ? fs0 : e.x) : fp0;
    float a1 = type == 0 ? (rank < 31 ? fs1 : e.y) : fp1;
    if (k < m) {
      on[k * 2 + cmi] = w2 * a1;                       // d W1[k][masked]
      on[k * 2 + cui] = 0.f;
      on[2 * m + k] = w2 * a0;                         // d b1[k]
      on[2 * m + m + cui * m + k] = fmaf(w1, a1, b1 * a0);   // d W2[transformed][k]
      on[2 * m + m + cmi * m + k] = 0.f;
    }
    if (net == 0 && lane < 8) {
      // 0,1: ActNorm.s[c]; 2,3: ActNorm.t[c]; 4,5: s.b2[c]; 6,7: t.b2[c]      scalar sums: [sas_m sat_m sas_u sat_u sb2s sb2t]
      const float* rs = Hs + f * FLOW_SEG_RS;
      float* out = outb + (int64_t)f * p.per_flow;
      const int qd = lane >> 1, c = lane & 1;
      const bool masked = c == cmi;
      const int src = qd == 0 ? (masked ? 0 : 2) : qd == 1 ? (masked ? 1 : 3) : qd == 2 ? 4 : 5;
      float a = rs[132 + src];
      if (qd >= 2 && masked) a = 0.f;
      if (qd == 2) out[2 * m + m + 2 * m + c] = a;
      else if (qd == 3) out[half + 2 * m + m + 2 * m + c] = a;
      else if (qd == 0) out[2 * half + c] = a;
      else out[2 * half + C + c] = a;
    }
  }
}

// ---------------------------------------------------------------- ActNorm data-dependent init
// z state lives in X[n] (pre-ActNorm output of the previous coupling).  One pass per flow.
template <int C>
__global__ void __launch_bounds__(256) k_flow_init_pass(FlowP p, int f, double* stats) {
  extern __shared__ float sp[];
  const float* par = p.params + p.off_flow;
  const int PF = (int)p.P_flow + 2 * C;
  for (int i = threadIdx.x; i < PF; i += blockDim.x) sp[i] = par[i];
  __syncthreads();
  int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int m = p.m, half = 2 * m * C + m + C;
  float zc[C];
  bool live = n < p.N;
#pragma unroll
  for (int c = 0; c < C; c++) zc[c] = 0.f;
  if (live) {
    float z[C];
    const float* lin = sp + p.P_flow;
    if (f == 0) {
#pragma unroll
      for (int c = 0; c < C; c++)
        z[c] = mm_fwd(coord(p.g, n, c) * lin[c] + lin[C + c], p.fc.nmin[c], p.fc.nmax[c], p.fc.new_min, p.fc.new_max);
    } else {
      const float* an = sp + (int64_t)(f - 1) * p.per_flow + 2 * half;   // ActNorm f-1, already initialised
      float4 v = *reinterpret_cast<const float4*>(p.X + n * 4);
      float zz[3] = {v.x, v.y, v.z};
#pragma unroll
      for (int c = 0; c < C; c++) z[c] = fmaf(zz[c], expf(an[c]), an[C + c]);
    }
    const float* w = sp + (int64_t)f * p.per_flow;
    float zm[C], so[C], to[C];
    bool b[C];
#pragma unroll
    for (int c = 0; c < C; c++) {
      b[c] = p.fc.masks[f * C + c] != 0; zm[c] = b[c] ? z[c] : 0.f;
      so[c] = w[m * C + m + C * m + c]; to[c] = w[half + m * C + m + C * m + c];
    }
    for (int k = 0; k < m; k++) {
      float ps = w[m * C + k], pt = w[half + m * C + k];
#pragma unroll
      for (int c = 0; c < C; c++) { ps = fmaf(w[k * C + c], zm[c], ps); pt = fmaf(w[half + k * C + c], zm[c], pt); }
      float hs = fmaxf(ps, 0.f), ht = fmaxf(pt, 0.f);
#pragma unroll
      for (int c = 0; c < C; c++) {
        so[c] = fmaf(w[m * C + m + c * m + k], hs, so[c]);
        to[c] = fmaf(w[half + m * C + m + c * m + k], ht, to[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < C; c++) {
      float s = p.tanh_out ? p.out_scale * tanhf(so[c]) : so[c], t = p.tanh_out ? p.out_scale * tanhf(to[c]) : to[c];
      zc[c] = b[c] ? z[c] : fmaf(z[c], expf(s), t);
    }
    *reinterpret_cast<float4*>(p.X + n * 4) = make_float4(zc[0], zc[1], C > 2 ? zc[2] : 0.f, 1.f);
  }
  // block sums of z and z^2 in double, then one atomic per block and statistic
  __shared__ double red[2 * 3][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int c = 0; c < C; c++) {
    double a = live ? (double)zc[c] : 0.0, q = a * a;
    for (int off = 16; off > 0; off >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, off);
      q += __shfl_xor_sync(0xffffffffu, q, off);
    }
    if (lane == 0) { red[c][warp] = a; red[3 + c][warp] = q; }
  }
  __syncthreads();
  if (threadIdx.x < 2 * C) {
    int c = threadIdx.x % C, which = threadIdx.x / C;
    double a = 0.0;
    for (int i = 0; i < 8; i++) a += red[which * 3 + c][i];
    atomicAdd(&stats[which * C + c], a);
  }
}

template <int C>
__global__ void k_flow_init_set(FlowP p, int f, const double* stats, float* params) {
  // s = -log(std + 1e-6) (unbiased std), t = -mean * exp(s)   (normflows ActNorm.forward, first call)
  int c = threadIdx.x;
  if (c >= C) return;
  const int m = p.m, half = 2 * m * C + m + C;
  double n = (double)p.N;
  double mean = stats[c] / n;
  double var = (stats[C + c] - stats[c] * stats[c] / n) / (n - 1.0);
  if (var < 0.0) var = 0.0;
  float sd = (float)sqrt(var);
  float s = -logf(sd + 1e-6f);
  float t = -(float)mean * expf(s);
  float* an = params + p.off_flow + (int64_t)f * p.per_flow + 2 * half;
  an[c] = s;
  an[C + c] = t;
}

// ---------------------------------------------------------------- learn_flow_identity loss
// loss = mean over N*C of (grid - flow_net(grid))^2  (SE("mean"), path_connected_net.py:172,223)
template <int C>
__global__ void __launch_bounds__(256) k_identity_loss(FlowP p, float* dX, float* lossp) {
  const int s = blockIdx.x, o = blockIdx.y;
  const int64_t r0 = (int64_t)s * p.chunk, r1 = r0 + p.chunk < p.N ? r0 + p.chunk : p.N;
  const float inv = 1.0f / ((float)p.N * (float)C);
  float acc = 0.f;
  for (int64_t n = r0 + threadIdx.x; n < r1; n += 256) {
    float4 v = *reinterpret_cast<const float4*>(p.X + ((int64_t)o * p.N + n) * 4);
    float xd[3] = {v.x, v.y, v.z};
    float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < C; c++) {
      float e = coord(p.g, n, c) - xd[c];
      acc = fmaf(e, e, acc);
      d[c] = -2.f * e * inv;
    }
    *reinterpret_cast<float4*>(dX + ((int64_t)o * p.N + n) * 4) = make_float4(d[0], d[1], d[2], 0.f);
  }
  __shared__ float red[8];
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f;
    for (int i = 0; i < 8; i++) a += red[i];
    lossp[s * p.O + o] = a * inv;
  }
}

// ======================================================================= launchers
static FlowP make_p(const awb_prior* h, const float* params, const awb_grid_spec* g, const Workspace& ws) {
  const Layout& L = h->lay;
  FlowP p = {};
  p.g.mode = g->mode; p.g.B = g->B; p.g.H = g->H; p.g.W = g->W; p.g.C = L.C;
  p.g.t0 = g->t0; p.g.t_step = g->t_step; p.g.grid = g->grid; p.g.row0 = (uint32_t)ws.row0;
  p.fc = h->fc;
  p.params = params; p.P = L.P; p.off_flow = L.off_flow; p.P_flow = L.P_flow; p.per_flow = L.per_flow;
  p.off_lin = L.off_lin;
  p.C = L.C; p.F = L.F; p.m = L.m; p.tanh_out = h->desc.flow_tanh; p.use_linear = 1; p.out_scale = h->fc.out_scale; p.inv_out_scale = 1.f / h->fc.out_scale;
  p.N = ws.N;
  p.X = ws.X; p.zin = nullptr; p.deformed = nullptr; p.dX = ws.dX; p.fpart = ws.fpart;
  p.chunk = split_chunk(p.N); p.O = h->desc.n_objects; p.rounds = 1; p.rounds1 = 0; p.dz_smem = 0; p.dzp_g = nullptr;
  p.tab = ws.flowtab; p.segscr = nullptr; p.dgrid = nullptr;
  return p;
}

// C = 2 priors can run the segment-table kernels.  Default (awb_prior_set_flow_eval mode 0): tensor-path handles do, fp32
// handles keep the unit loops -- the fp32 path is the parity anchor and evaluates the MLPs in the reference's order of
// operations; the tables reassociate the sums (differences at the 1e-7 level, tests/test_gpu_flow.py).
static size_t flow_seg_bwd_smem(const awb_prior* h, int T, int64_t chunk_in_smem) {
  const size_t hist = (size_t)FLOW_SEG_ROWS * T, rows = (size_t)h->lay.F * FLOW_SEG_RS;      // the region is reused for the summed rows
  return sizeof(float) * ((size_t)h->lay.F * (FLOW_TAB + 4) + 64 + 2 * (size_t)FLOW_PB * T * 4 + (hist > rows ? hist : rows) +
                          2 * (size_t)chunk_in_smem);
}
bool flow_seg_capable(const awb_prior* h) {
  return h->desc.kind == AWB_KIND_FLOW_ICNN && h->lay.C == 2 && h->lay.m <= 32 && flow_seg_bwd_smem(h, FLOW_BWD_T, 0) <= 220 * 1024;
}
bool flow_seg_path(const awb_prior* h) {
  // (the segment kernels are specialised for the standard couplings s, t = tanh(MLP); anything else keeps the unit loops)
  if (!flow_seg_capable(h) || h->flow_eval == 1 || !h->desc.flow_tanh || h->fc.out_scale != 1.f) return false;
  return h->flow_eval == 2 || h->desc.precision == AWB_PREC_F16;
}
int64_t flow_seg_scratch_floats(const awb_prior* h, int S) {
  return flow_seg_capable(h) ? (int64_t)S * h->desc.n_objects * h->lay.F * 8 * FLOW_SEG_RS : 0;
}
// C = 3: forward tables for the flows with one masked coordinate (the backward keeps the unit loops)
bool flow_seg3_capable(const awb_prior* h) { return h->desc.kind == AWB_KIND_FLOW_ICNN && h->lay.C == 3 && h->lay.m <= 32; }
bool flow_seg3_path(const awb_prior* h) {
  if (!flow_seg3_capable(h) || h->flow_eval == 1 || !h->desc.flow_tanh || h->fc.out_scale != 1.f) return false;
  return h->flow_eval == 2 || h->desc.precision == AWB_PREC_F16;
}
int64_t flow_tab_floats(const awb_prior* h) {
  if (flow_seg3_capable(h)) return (int64_t)h->desc.n_objects * h->lay.F * FLOW_TAB3;
  return flow_seg_capable(h) ? (int64_t)h->desc.n_objects * h->lay.F * FLOW_TAB : 0;
}

int flow_forward(const awb_prior* h, const float* params, const awb_grid_spec* g, const Workspace& ws,
                 float* deformed, cudaStream_t st, bool use_linear) {
  FlowP p = make_p(h, params, g, ws);
  p.use_linear = use_linear ? 1 : 0;
  p.zin = ws.flowz;
  p.deformed = deformed;
  // The forward has no per-CTA partials, so the number of CTAs is free: k CTAs of 128 threads per SM (latency hiding: the
  // kernel needs 47 registers), each with one or two full rounds of FLOW_P pixels per thread and a one-pixel remainder
  // round, sized so that every SM gets the same number of pixels.
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
  FlowGeo geo;
  const bool seg = flow_seg_path(h) && p.tab;
  const bool seg3 = flow_seg3_path(h) && p.tab;
  if (h->lay.C == 3 && !seg3) p.tab = nullptr;      // k_flow_fwd<3> takes a non-null table pointer as "tables are built"
  geo.T = (seg || seg3) ? 256 : 128;        // segment kernels: the per-CTA table staging is amortised over twice the pixels
  int64_t per_sm = (p.N * h->desc.n_objects + sms - 1) / sms;
  int k = (int)((per_sm + FLOW_P * geo.T / 2) / (FLOW_P * geo.T));
  if (k < 1) k = 1;
  if (k > 8) k = 8;
  int64_t n_cta = (int64_t)sms * k / h->desc.n_objects;
  if (n_cta < 1) n_cta = 1;
  geo.chunk = (p.N + n_cta - 1) / n_cta;
  if (geo.chunk < 32) geo.chunk = 32;
  geo.S = (int)((p.N + geo.chunk - 1) / geo.chunk);
  if (geo.chunk < geo.T) geo.T = (int)round_up(geo.chunk, 32);
  geo.R = (int)(geo.chunk / ((int64_t)FLOW_P * geo.T));
  p.chunk = geo.chunk; p.rounds = geo.R;
  p.rounds1 = (int)((geo.chunk - (int64_t)geo.R * FLOW_P * geo.T + geo.T - 1) / geo.T);
  size_t smem = sizeof(float) * ((size_t)h->lay.F * (h->lay.C == 2 ? FlowPack<2>::flow_stride(h->lay.m) : FlowPack<3>::flow_stride(h->lay.m)) + 2 * h->lay.C);
  dim3 grid(geo.S, h->desc.n_objects);
  if (seg) {
    smem = sizeof(float) * ((size_t)h->lay.F * (FLOW_TAB_FWD + 4) + 4);
    AWB_LAUNCH(PK_FLOW_FWD, st, k_flow_tables<<<dim3(h->lay.F, h->desc.n_objects), 64, 0, st>>>(p));
    AWB_CUDA(cudaFuncSetAttribute(k_flow_fwd_seg, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    AWB_LAUNCH(PK_FLOW_FWD, st, k_flow_fwd_seg<<<grid, geo.T, smem, st>>>(p));
  } else if (h->lay.C == 2) {
    AWB_CUDA(cudaFuncSetAttribute(k_flow_fwd<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    AWB_LAUNCH(PK_FLOW_FWD, st, k_flow_fwd<2><<<grid, geo.T, smem, st>>>(p));
  } else {
    if (seg3) {
      smem += sizeof(float) * (2 + (size_t)h->lay.F * FLOW_TAB3);
      AWB_LAUNCH(PK_FLOW_FWD, st, k_flow_tables3<<<dim3(h->lay.F, h->desc.n_objects), 64, 0, st>>>(p));
    }
    AWB_CUDA(cudaFuncSetAttribute(k_flow_fwd<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    AWB_LAUNCH(PK_FLOW_FWD, st, k_flow_fwd<3><<<grid, geo.T, smem, st>>>(p));
  }
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int flow_inverse(const awb_prior* h, const float* params, const awb_grid_spec* g, float* out, cudaStream_t st) {
  Workspace none = {};
  none.N = (int64_t)g->B * g->H * g->W;
  FlowP p = make_p(h, params, g, none);
  const int PF = (int)(h->lay.P_flow + 2 * h->lay.C);
  size_t smem = sizeof(float) * PF;
  dim3 grid((unsigned)((p.N + 255) / 256), h->desc.n_objects);
  if (h->lay.C == 2) {
    AWB_CUDA(cudaFuncSetAttribute(k_flow_inv<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    AWB_LAUNCH(PK_FLOW_FWD, st, k_flow_inv<2><<<grid, 256, smem, st>>>(p, out));
  } else {
    AWB_CUDA(cudaFuncSetAttribute(k_flow_inv<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    AWB_LAUNCH(PK_FLOW_FWD, st, k_flow_inv<3><<<grid, 256, smem, st>>>(p, out));
  }
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

// shared memory of k_flow_bwd without / with the running gradient of the CTA's pixel range
static size_t flow_bwd_smem_base(const awb_prior* h) {
  const int C = h->lay.C;
  return sizeof(float) * ((size_t)h->lay.F * (C == 2 ? FlowBwdPack<2>::flow_stride() : FlowBwdPack<3>::flow_stride()) + 2 * FLOW_RED_FLOATS +
                          2 * (size_t)FLOW_PB * flow_save_floats(C) * FLOW_BWD_T);
}
bool flow_bwd_dz_in_smem(const awb_prior* h, int64_t N) {
  const int C = h->lay.C;
  const size_t dz = sizeof(float) * (size_t)split_chunk(N) * C * (C == 3 ? 2 : 1);
  return flow_bwd_smem_base(h) + dz <= 200 * 1024;
}

int flow_backward(const awb_prior* h, const float* params, const awb_grid_spec* g, const Workspace& ws,
                  cudaStream_t st, bool use_linear, float* dgrid) {
  FlowP p = make_p(h, params, g, ws);
  p.use_linear = use_linear ? 1 : 0;
  p.zin = ws.flowz;
  p.dgrid = dgrid;
  if (!p.zin) { set_error("flow backward needs a training workspace"); return AWB_ERR_WORKSPACE; }
  if (dgrid && (!use_linear || h->desc.n_objects != 1)) { set_error("internal: dgrid needs one object and the 1x1 conv"); return AWB_ERR_INVALID; }
  if (h->lay.m > 32) { set_error("flow MLP width must be <= 32"); return AWB_ERR_UNSUPPORTED; }
  const int C = h->lay.C;
  for (int f = 0; f < h->lay.F; f++) {
    int mb = 0;
    for (int c = 0; c < C; c++) mb |= h->fc.masks[f * C + c] != 0 ? 1 << c : 0;
    if (mb < 1 || mb > (1 << C) - 2) {
      set_error("flow %d has a degenerate coupling mask (all or no component masked): not trainable", f);
      return AWB_ERR_UNSUPPORTED;
    }
  }
  // T threads; full rounds of FLOW_PB pixels per thread, then the remainder of the range in rounds of one pixel per thread
  // (2080 rows = 2 x 1024 + 32: a third full round for 32 pixels would cost its warp 50 %)
  FlowGeo geo;
  geo.S = n_splits(p.N); geo.chunk = split_chunk(p.N);
  geo.T = (int)(geo.chunk < FLOW_BWD_T ? round_up(geo.chunk, 32) : FLOW_BWD_T);
  geo.R = (int)(geo.chunk / ((int64_t)FLOW_PB * geo.T));
  p.chunk = geo.chunk; p.rounds = geo.R;
  p.rounds1 = (int)((geo.chunk - (int64_t)geo.R * FLOW_PB * geo.T + geo.T - 1) / geo.T);
  p.dz_smem = flow_bwd_dz_in_smem(h, p.N) ? 1 : 0;
  p.dzp_g = ws.flowd;
  if (!p.dz_smem && C == 3 && !p.dzp_g) { set_error("flow backward: workspace lacks the pass scratch"); return AWB_ERR_WORKSPACE; }
  size_t smem = flow_bwd_smem_base(h) + (p.dz_smem ? sizeof(float) * (size_t)geo.chunk * C * (C == 3 ? 2 : 1) : 0);
  dim3 grid(geo.S, h->desc.n_objects);
  if (flow_seg_path(h) && p.tab) {
    geo.T = FLOW_BWD_T;          // the segment kernel always runs 256 threads (idle ones for tiny ranges)
    const int64_t wl = (geo.chunk + FLOW_BWD_T / 32 - 1) / (FLOW_BWD_T / 32);      // pixels of one warp's block
    geo.R = (int)(wl / (32 * FLOW_PB));
    p.rounds = geo.R;
    p.rounds1 = (int)((wl - (int64_t)geo.R * 32 * FLOW_PB + 31) / 32);
    p.dz_smem = flow_seg_bwd_smem(h, geo.T, geo.chunk) <= 220 * 1024 ? 1 : 0;
    smem = flow_seg_bwd_smem(h, geo.T, p.dz_smem ? geo.chunk : 0);
    p.segscr = ws.flowseg;
    if (!p.segscr) { set_error("flow backward: workspace lacks the segment scratch"); return AWB_ERR_WORKSPACE; }
    auto seg = [&](auto kernel) -> int {
      AWB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      AWB_LAUNCH(PK_FLOW_BWD, st, AWB_CUDA(launch_ex(kernel, grid, dim3(geo.T), smem, st, true, p)));
      return AWB_OK;
    };
    int rc = p.dz_smem ? (dgrid ? seg(k_flow_bwd_seg<true, true>) : seg(k_flow_bwd_seg<true, false>))
                       : (dgrid ? seg(k_flow_bwd_seg<false, true>) : seg(k_flow_bwd_seg<false, false>));
    if (rc) return rc;
  } else {
    auto unit = [&](auto kernel) -> int {
      AWB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      AWB_LAUNCH(PK_FLOW_BWD, st, kernel<<<grid, geo.T, smem, st>>>(p));
      return AWB_OK;
    };
    int rc = C == 2 ? (dgrid ? unit(k_flow_bwd<2, true>) : unit(k_flow_bwd<2, false>))
                    : (dgrid ? unit(k_flow_bwd<3, true>) : unit(k_flow_bwd<3, false>));
    if (rc) return rc;
  }
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int flow_identity_loss(const awb_prior* h, const awb_grid_spec* g, const Workspace& ws, cudaStream_t st) {
  FlowP p = make_p(h, nullptr, g, ws);
  dim3 grid(n_splits(p.N), h->desc.n_objects);
  if (h->lay.C == 2) AWB_LAUNCH(PK_OUT_LOSS, st, k_identity_loss<2><<<grid, 256, 0, st>>>(p, ws.dX, ws.lossp));
  else AWB_LAUNCH(PK_OUT_LOSS, st, k_identity_loss<3><<<grid, 256, 0, st>>>(p, ws.dX, ws.lossp));
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int flow_actnorm_init(const awb_prior* h, float* params, const awb_grid_spec* g, const Workspace& ws,
                      cudaStream_t st) {
  if (h->desc.n_objects != 1) { set_error("ActNorm init is per object: call it on single-object handles"); return AWB_ERR_UNSUPPORTED; }
  FlowP p = make_p(h, params, g, ws);
  const int C = h->lay.C;
  const int PF = (int)(h->lay.P_flow + 2 * C);
  size_t smem = sizeof(float) * PF;
  double* stats = (double*)ws.lossp;            // 2*C doubles of scratch (lossp is 256-byte aligned, >= 8 floats)
  if (C == 2) AWB_CUDA(cudaFuncSetAttribute(k_flow_init_pass<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  else AWB_CUDA(cudaFuncSetAttribute(k_flow_init_pass<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  unsigned blocks = (unsigned)((p.N + 255) / 256);
  for (int f = 0; f < h->lay.F; f++) {
    AWB_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * 6, st));
    if (C == 2) {
      AWB_LAUNCH(PK_MISC, st, k_flow_init_pass<2><<<blocks, 256, smem, st>>>(p, f, stats));
      AWB_LAUNCH(PK_MISC, st, k_flow_init_set<2><<<1, 32, 0, st>>>(p, f, stats, params));
    } else {
      AWB_LAUNCH(PK_MISC, st, k_flow_init_pass<3><<<blocks, 256, smem, st>>>(p, f, stats));
      AWB_LAUNCH(PK_MISC, st, k_flow_init_set<3><<<1, 32, 0, st>>>(p, f, stats, params));
    }
  }
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

}  // namespace awb
