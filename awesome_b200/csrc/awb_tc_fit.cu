// Fused ICNN fit step on the Blackwell tensor path (AWB_PREC_F16): ONE persistent kernel does, per
// 128-pixel tile, coordinate generation -> input layer -> L hidden layers -> output layer + sigmoid +
// loss -> full backward (data gradients and weight gradients), with
//   * every layer contraction (forward, dgrad, wgrad) on tcgen05.mma kind::f16 (fp16 operands, fp32
//     accumulation in TMEM), M = 128 pixels, N = K = 144 (130 hidden + skip/bias augmentation + pad);
//   * bias and skip connection folded into the contraction through the augmented K columns (x, 1);
//   * weights staged once per CTA in shared memory by TMA bulk copies (cp.async.bulk + mbarrier);
//   * activations never leaving the SM: TMEM -> registers (relu / relu-backward / loss) -> fp16
//     shared-memory operand tiles of the next contraction;
//   * weight gradients accumulated across all tiles of the CTA in TMEM (dW never touches HBM until
//     the single per-CTA partial write at the end, staged through shared memory and written with TMA
//     bulk stores); the 130 = 128 + 2 remainder rows/columns are covered by two N=16 side
//     contractions plus a handful of per-thread corner sums;
//   * loss / corner sums reduced with registers + one shared-memory pass (no atomics).
// The cross-CTA reduction + Adam/Adamax + clamp + plateau run in k_reduce_opt (awb_simt.cu).
//
// Pipeline (one tile in flight; shared memory holds the weights (81 KB) + 4 operand tiles (136 KB)):
//   epilogue warps (8) <-> issuer (1 elected lane) through two mbarriers; 2L+1 round trips per tile.
//   Everything that is not on the round-trip critical path runs in the shadow of the next
//   contraction: next tile's coordinates / target prefetch, corner sums, loss accumulation, the
//   relu masks of the backward epilogues (read from the stored activations before the wait).
//
// Shared-memory operand tiles use the SWIZZLE_NONE interleaved layout of awb_tc.cuh with 17 stored
// column chunks (136 columns); the 18th chunk of a K = 144 walk is redirected to a shared zero chunk
// through the per-instruction LBO field, and as an MN-major N = 144 operand it reads whatever follows
// (those accumulator columns, 136..143, are never read).  See DESIGN.md "tensor path".
#include <math.h>
#include <stdlib.h>

#include <type_traits>
#include <vector>

#include "awb_internal.cuh"
#include "awb_tc.cuh"

namespace awb {

namespace {
constexpr int H_ = 130, LD_ = 136, NPAD = 144;
constexpr int TILE_B = 17 * 2048;   // [17 chunks][128 rows][8 fp16]
constexpr int W_B = 17 * 2304;      // [17 chunks][144 rows][8 fp16]
constexpr int WIN_B = 2304;         // [1 chunk][144 rows][8 fp16]   input layer (K = 16: 2nd chunk = zero chunk)
constexpr int TX_B = 2048;          // [1 chunk][128 rows][8 fp16]   (x, y, (t), 1, 0...), double buffered
constexpr int ZERO_B = 2304;
constexpr int VEC_B = NPAD * 4;     // fp32 (w_o | s_o | b_o | 0)
constexpr int VEC16_B = NPAD * 2;   // the same vector as fp16 (operand of the packed delta_L product)
constexpr int NCG = 3;              // epilogue column groups per TMEM lane quadrant
constexpr int NEW = 4 * NCG;        // epilogue warps (3 per warp scheduler)
constexpr int NTHREADS = (NEW + 1) * 32;   // + 1 issuer warp
constexpr int XCHG_B = NCG * 128 * 4;
constexpr int XCHG2_B = (NCG - 1) * 128 * 3 * 4;   // input-layer coordinate-gradient partials (flow priors)
constexpr int TRACE_N = 256;        // clock stamps per CTA (debug timeline)
__host__ __device__ constexpr int img_bytes(int L) { return L * W_B + WIN_B + VEC_B + VEC16_B; }
__host__ __device__ constexpr int smem_bytes(int L) {
  return (L + 2) * TILE_B + img_bytes(L) + 2 * TX_B + ZERO_B + XCHG_B + XCHG2_B + 64;
}
}  // namespace

int tc_image_bytes(int L) { return (int)round_up(img_bytes(L), 256); }

// ------------------------------------------------------------------ weight image (fp32 arena -> fp16 UMMA tiles)
__global__ void k_pack_tc(const float* __restrict__ params, uint8_t* __restrict__ img, const int32_t* __restrict__ tcmap,
                          int n_elems, int L, int64_t P, int64_t img_stride) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int o = blockIdx.y;
  if (i >= n_elems) return;
  int32_t src = tcmap[i];
  float v = src >= 0 ? params[(int64_t)o * P + src] : 0.f;
  const int n_half = (L * W_B + WIN_B) / 2;
  uint8_t* base = img + (int64_t)o * img_stride;
  if (i < n_half) reinterpret_cast<__half*>(base)[i] = __float2half_rn(v);
  else if (i < n_half + NPAD) reinterpret_cast<float*>(base + 2 * n_half)[i - n_half] = v;
  else reinterpret_cast<__half*>(base + 2 * n_half + VEC_B)[i - n_half - NPAD] = __float2half_rn(v);
}

struct TcP {
  GridDev g;
  const uint8_t* img; int64_t img_stride;
  const float* target;
  LossCoef loss[16];
  float scale[16];
  float* part; int64_t sSplit, G, aug_in, aug_layer, aug_out;
  float* lossp; int O;
  float* logits;
  int64_t N; int n_tiles; int mode;
  unsigned long long* trace;
  int trace_serial;
  const float* amax;   // optional device [O]: max |dlogits| per object; sets the fp16 loss scale of the upstream-gradient mode
  const float* X;   // optional [O][N][4]: coordinates produced by the flow (x, y, t, 1) instead of the generated grid
  float* dX;        // optional [O][N][4]: gradient w.r.t. those coordinates (consumed by the flow backward)
  // WL only: weight map and ignore label per object; the fp16 loss scale then comes from max |w| over the kept pixels
  // (wamax, device [O]) times max |coef| (coef_max)
  LossPix pix[16];
  float coef_max[16];
  const float* wamax;
};

__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
// (lo, hi) fp32 -> packed fp16 pair with relu, one instruction (cvt.rn.relu.f16x2.f32; NaN -> canonical NaN like fmaxf's
// operand order would not matter here: the loss of a NaN row is flagged non-finite upstream)
__device__ __forceinline__ uint32_t pack2_relu(float a, float b) {
  uint32_t r;
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ uint32_t relu2(uint32_t u) {   // max(x, 0) on a packed fp16 pair
  __half2 h = *reinterpret_cast<__half2*>(&u);
  h = __hmax2(h, __float2half2_rn(0.f));
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t gt0_mask2(uint32_t u) {   // 0xFFFF per half that is > 0
  return __hgt2_mask(*reinterpret_cast<__half2*>(&u), __float2half2_rn(0.f));
}
__device__ __forceinline__ void st16(uint8_t* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  *reinterpret_cast<uint4*>(p) = make_uint4(a, b, c, d);
}
__device__ __forceinline__ float half_lo(uint32_t u) { return __low2float(*reinterpret_cast<__half2*>(&u)); }
__device__ __forceinline__ float half_hi(uint32_t u) { return __high2float(*reinterpret_cast<__half2*>(&u)); }
// pixel coordinates with 32-bit index arithmetic (N <= 2^30 is checked on the host)
// Out of line on purpose: the hot loop only carries the division-free linspace path; explicit grids, the notebooks'
// index grid and the padding rows of a last tile come here (the fused kernel's speed depends on its code footprint).
__device__ __noinline__ void row_coords(const GridDev g, uint32_t n, int C, float& x0, float& x1, float& x2) {
  n += g.row0;   // local -> global row
  const uint32_t hw = (uint32_t)g.H * (uint32_t)g.W;
  const uint32_t b = n / hw, r = n - b * hw;
  const uint32_t i = r / (uint32_t)g.W, j = r - i * (uint32_t)g.W;
  if (g.mode == AWB_GRID_EXPLICIT) {
    const float* base = g.grid + (size_t)b * C * hw + r;
    x0 = base[0]; x1 = base[hw]; x2 = C > 2 ? base[2 * (size_t)hw] : 0.f;
    return;
  }
  x2 = C > 2 ? g.t0 + (float)b * g.t_step : 0.f;
  if (g.mode == AWB_GRID_LINSPACE) { x0 = lin01((int)j, g.W); x1 = lin01((int)i, g.H); }
  else { x0 = (float)j / (float)g.W; x1 = (float)i / (float)g.H; }
}

__device__ __noinline__ float bce_logits(float y, float t) {   // BCEWithLogits, stable form; rare: kept out of the hot loop
  return fmaxf(y, 0.f) - y * t + log1pf(expf(-fabsf(y)));
}

// Sum of v[i] over the 32 lanes of a warp for 16 values at once: one butterfly round, then four
// reduce-scatter rounds; afterwards lane l holds the total of value (l & 15).  31 shuffles instead of 80.
__device__ __forceinline__ float warp_reduce_scatter16(float* v, int lane) {
#pragma unroll
  for (int k = 0; k < 16; k++) v[k] += __shfl_xor_sync(0xffffffffu, v[k], 16);
#pragma unroll
  for (int off = 8, n = 16; off >= 1; off >>= 1, n >>= 1) {
    const bool up = lane & off;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      if (k < n / 2) {
        const float send = up ? v[k] : v[k + n / 2];
        const float keep = up ? v[k + n / 2] : v[k];
        v[k] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
  }
  return v[0];
}

// FIT: forward + loss + backward + partials (else forward only, logits out); DX: the coordinates come from a flow and
// their gradient goes back to it; WL (with FIT): per-pixel loss weights and / or an ignore label, the weight fetched
// with the target.  Compile-time so that the forward-only and the plain ICNN instantiations carry
// neither the branches nor the live ranges (delta_0 words, coordinate-gradient sums) of the others.
template <int L, int C, bool FIT, bool DX, bool WL>
__global__ void __launch_bounds__(NTHREADS, 1) k_icnn_fit_tc(TcP p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  constexpr int NT = L + 2;
  constexpr int IMG = img_bytes(L);
  uint8_t* tiles = smem;                          // ZT[0..L-1], ZL, DT
  uint8_t* simg = smem + NT * TILE_B;             // W_1..W_L | WIN | vec | vec16
  uint8_t* stx = simg + IMG;                      // TX[2]
  uint8_t* szero = stx + 2 * TX_B;
  float* xchg = reinterpret_cast<float*>(szero + ZERO_B);          // [NCG][128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(szero + ZERO_B + XCHG_B + XCHG2_B);
  uint64_t* bar_e2m = bars;        // epilogue -> issuer (one arrival per epilogue warp)
  uint64_t* bar_m2e = bars + 1;    // tcgen05.commit -> epilogue
  uint64_t* bar_w = bars + 2;      // weight image landed (TMA tx bytes)
  uint64_t* bar_dbg = bars + 3;    // diagnostic build only: the issuer waits for every contraction group
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
  const float* wo = reinterpret_cast<const float*>(simg + L * W_B + WIN_B);
  const uint8_t* wo16 = simg + L * W_B + WIN_B + VEC_B;            // fp16 copy, 16 bytes per column chunk

  // Hardware warp 0 issues the contractions; hardware warps 1..12 are the epilogue warps.  `warp` is their logical index
  // 4 * column group + lane quadrant, with the quadrant = hardware warp % 4 (the TMEM lanes a warp may touch).
  const int hwarp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int warp = hwarp == 0 ? NEW : ((((hwarp - 1) >> 2) << 2) | (hwarp & 3));
  const int o = blockIdx.y;
  const bool issuer_warp = warp == NEW;
  // In-kernel timeline (clock64 stamps of one epilogue thread and of the issuer): compiled in only for the diagnostic
  // builds (-DAWB_TC_TRACE_BUILD / -DAWB_TC_SERIAL, scripts/trace_tc.py) -- the stamps' predicated stores sit inside the
  // issuer's and the epilogue's hot loops.
#if defined(AWB_TC_TRACE_BUILD) || defined(AWB_TC_SERIAL)
  unsigned long long* trace = p.trace ? p.trace + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * TRACE_N : nullptr;
  int tr_n = 0;
#define AWB_TR()                                                            \
  do {                                                                      \
    if (trace && lane == 0 && (warp == 0 || issuer_warp) && tr_n < 120)        \
      trace[(issuer_warp ? TRACE_N / 2 : 0) + tr_n++] = clock64();          \
  } while (0)
#else
  constexpr unsigned long long* trace = nullptr;
#define AWB_TR() do {} while (0)
#endif

  if (trace && warp == 0 && lane == 0) {                       // kernel entry (SM cycles and wall-clock ns)
    trace[120] = clock64();
    unsigned long long ns;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    trace[125] = ns;
  }
  // ---- one-time setup
  if (threadIdx.x == 0) { tc::mbar_init(bar_e2m, NEW); tc::mbar_init(bar_m2e, 1); tc::mbar_init(bar_w, 1); tc::mbar_init(bar_dbg, 1); tc::mbar_fence_init(); }
  for (int i = threadIdx.x * 16; i < ZERO_B; i += NTHREADS * 16) *reinterpret_cast<uint4*>(szero + i) = make_uint4(0, 0, 0, 0);
  __syncthreads();
  if (issuer_warp) tc::tmem_alloc<512>(tmem_slot);
  // Everything above overlaps the tail of the previous kernel in the stream (programmatic dependent launch);
  // from here on this kernel reads what that kernel wrote (weight image, unaries, flow coordinates).
  grid_dep_wait();
  grid_dep_launch();
  if (issuer_warp) {
    if (lane == 0) {
      const uint8_t* src = p.img + (int64_t)o * p.img_stride;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc::smem_u32(bar_w)), "r"((uint32_t)IMG) : "memory");
      for (int off = 0; off < IMG; off += 16384) {
        uint32_t sz = IMG - off < 16384 ? IMG - off : 16384;
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(tc::smem_u32(simg + off)), "l"(src + off), "r"(sz), "r"(tc::smem_u32(bar_w)) : "memory");
      }
    }
  }
  tc::fence_async_smem();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tbase = *tmem_slot;

  constexpr uint32_t T_ACC = 0;
  auto T_DW = [](int i) { return (uint32_t)(144 * i); };                       // i = 1..L
  auto T_PB = [](int i) { return (uint32_t)(144 * (L + 1) + 16 * (i - 1)); };  // i = 1..L
  constexpr uint32_t T_GIN = 144 * (L + 1) + 16 * L, T_GO = T_GIN + 16;
  constexpr uint32_t T_DX = T_GO + 16;      // flow priors: delta_0 * W_in = gradient reaching the coordinates through the input layer
  static_assert(T_DX + 16 <= 512, "TMEM budget");

  auto tile_ptr = [&](int t) { return tiles + t * TILE_B; };       // t < L: ZT[t]; L: ZL; L+1: DT
  auto dbuf = [&](int i) { return tile_ptr(((L - i) & 1) ? L : L + 1); };      // delta_i lives in DT / ZL alternately

  const int n_my = (p.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  constexpr bool fit = FIT;

  if (issuer_warp) {
    // =========================================================== MMA issuer (one elected lane)
    if (lane == 0) {
      tc::mbar_wait(bar_w, 0);
      uint32_t ph = 0;
      const uint32_t zero_a = tc::smem_u32(szero);
      const uint32_t a_tx0 = tc::smem_u32(stx), a_win = tc::smem_u32(simg + L * W_B);
      auto w_addr = [&](int i) { return tc::smem_u32(simg + (i - 1) * W_B); };
      auto t_addr = [&](uint8_t* t) { return tc::smem_u32(t); };
      // K-major A (R=128) x K-major/MN-major B (R=144) over K = 144 (9 steps), N = 144.  Descriptor bases once per
      // contraction -- prepared BEFORE the issuer waits for the epilogue warps, so that only the adds and the
      // instructions themselves sit between its wake-up and the tensor pipe -- and per instruction only the
      // start-address field advances (byte step >> 4).
      struct K144 { tc::DescLH a0, a8, b0, b8; uint32_t binc, idesc; };
      auto prep_k144 = [&](uint32_t a, uint32_t b, bool b_mn) {
        K144 d;
        d.idesc = tc::make_idesc(128, 144, 0, b_mn ? 1 : 0);
        d.a0 = tc::make_desc_lh(a, 2048, 128);
        d.a8 = tc::make_desc_lh(a + 8 * 4096, zero_a - (a + 8 * 4096), 128);     // 18th chunk -> zero chunk
        d.b0 = b_mn ? tc::make_desc_lh(b, 128, 2304) : tc::make_desc_lh(b, 2304, 128);
        d.b8 = b_mn ? tc::make_desc_lh(b + 8 * 256, 128, 2304) : tc::make_desc_lh(b + 8 * 4608, zero_a - (b + 8 * 4608), 128);
        d.binc = b_mn ? 256 / 16 : 4608 / 16;
        return d;
      };
      auto issue_k144 = [&](uint32_t dcol, const K144& d) {
#pragma unroll
        for (int k = 0; k < 8; k++)
          tc::umma_f16_lh(tbase + dcol, d.a0.lo + k * (4096 / 16), d.a0.hi, d.b0.lo + k * d.binc, d.b0.hi, d.idesc, k > 0);
        tc::umma_f16_lh(tbase + dcol, d.a8.lo, d.a8.hi, d.b8.lo, d.b8.hi, d.idesc, 1);
      };
      auto mma_k144 = [&](uint32_t dcol, uint32_t a, uint32_t b, bool b_mn) { issue_k144(dcol, prep_k144(a, b, b_mn)); };
      // MN-major A window [0,128) x MN-major B, K = 128 pixels (8 steps); b_sbo = byte distance of B's 2nd N chunk
      auto mma_px = [&](uint32_t dcol, uint32_t a, uint32_t b, uint32_t b_sbo, int N, bool acc) {
#ifdef AWB_TC_NO_STRIPS
        if (N == 16) return;      // timing experiment only (wrong gradients): upper bound of what the N = 16 strips cost
#endif
        const uint32_t idesc = tc::make_idesc(128, N, 1, 1);
        const tc::DescLH a0 = tc::make_desc_lh(a, 128, 2048), b0 = tc::make_desc_lh(b, 128, b_sbo);
#pragma unroll
        for (int k = 0; k < 8; k++)
          tc::umma_f16_lh(tbase + dcol, a0.lo + k * (256 / 16), a0.hi, b0.lo + k * (256 / 16), b0.hi, idesc,
                          (acc || k > 0) ? 1u : 0u);
      };
      // coordinate gradient through the input layer (flow priors): DXIN[128 x 16] = delta_0[128 x 144] * WIN[144 x 16] --
      // A like every K-major delta tile (18th chunk -> zero chunk), B = the WIN bytes read MN-major (N chunk 1 = zero chunk)
      auto mma_dx = [&](uint32_t a) {
        const uint32_t idesc = tc::make_idesc(128, 16, 0, 1);
        const tc::DescLH a0 = tc::make_desc_lh(a, 2048, 128), a8 = tc::make_desc_lh(a + 8 * 4096, zero_a - (a + 8 * 4096), 128);
        const tc::DescLH b0 = tc::make_desc_lh(a_win, 128, zero_a - a_win);
#pragma unroll
        for (int k = 0; k < 8; k++)
          tc::umma_f16_lh(tbase + T_DX, a0.lo + k * (4096 / 16), a0.hi, b0.lo + k * (256 / 16), b0.hi, idesc, k > 0);
        tc::umma_f16_lh(tbase + T_DX, a8.lo, a8.hi, b0.lo + 8 * (256 / 16), b0.hi, idesc, 1);
      };
      // input layer of a tile: ACC = TX[128x16] * WIN^T   (both operands: one stored K chunk + the zero chunk)
      const tc::DescLH in_b = tc::make_desc_lh(a_win, zero_a - a_win, 128);
      auto mma_input = [&](uint32_t a_tx) {
        const tc::DescLH in_a = tc::make_desc_lh(a_tx, zero_a - a_tx, 128);
        tc::umma_f16_lh(tbase + T_ACC, in_a.lo, in_a.hi, in_b.lo, in_b.hi, tc::make_idesc(128, 144, 0, 0), 0);
      };
      // Diagnostic build (-DAWB_TC_SERIAL, see scripts/trace_tc.py) with AWB_TC_TRACE=2: a commit + wait + clock stamp
      // after every contraction group gives the true duration of each.  Compiled out otherwise: even a never-taken
      // branch between the groups costs the issuing thread ~6 % of the kernel (measured).
#ifdef AWB_TC_SERIAL
      uint32_t phd = 0;
      const bool serial = trace && p.trace_serial;
      auto dbg = [&]() {
        if (serial) { tc::umma_commit(bar_dbg); tc::mbar_wait(bar_dbg, phd); phd ^= 1; AWB_TR(); }
      };
#else
      auto dbg = []() {};
#endif
      // prologue: input layer of the first tile
      tc::mbar_wait(bar_e2m, ph); ph ^= 1;
      tc::fence_after_sync();
      mma_input(a_tx0);
      tc::umma_commit(bar_m2e);
      AWB_TR();
      for (int it = 0; it < n_my; it++) {
        const bool acc = it > 0;
        const bool more = it + 1 < n_my;
        const uint32_t a_tx = a_tx0 + (it & 1) * TX_B, a_txn = a_tx0 + ((it + 1) & 1) * TX_B;
        if constexpr (!FIT) {
          for (int s = 1; s <= L + 1; s++) {
            tc::mbar_wait(bar_e2m, ph); ph ^= 1;
            tc::fence_after_sync();
            if (s <= L) mma_k144(T_ACC, t_addr(tile_ptr(s - 1)), w_addr(s), false);
            else if (more) mma_input(a_txn);
            tc::umma_commit(bar_m2e);
          }
        } else
        for (int s = 1; s <= 2 * L + 1; s++) {
          // operands of the stage's first contraction are known before the epilogue warps arrive
          const int i = s <= L ? s : L - (s - (L + 1));                           // forward layer s / delta_i just written
          const uint32_t d = t_addr(s <= L ? tile_ptr(s - 1) : dbuf(i > 0 ? i : 0));
          const K144 first = prep_k144(d, w_addr(i > 0 ? i : 1), s > L);
          tc::mbar_wait(bar_e2m, ph); ph ^= 1;
          tc::fence_after_sync();
          AWB_TR();
          if (s <= L) {
            issue_k144(T_ACC, first);                                             // forward layer s
            dbg();
            tc::umma_commit(bar_m2e);
          } else if (s <= 2 * L) {
            const uint32_t zprev = t_addr(tile_ptr(i - 1));
            issue_k144(T_ACC, first);                                             // dgrad_i: ACC = delta_i * W_i
            dbg();
            if (i == L) { mma_px(T_GO, t_addr(tile_ptr(L)), d + 16 * 2048, 2048, 16, acc); dbg(); }   // z_L^T * [d128 d129 dy ..]
            tc::umma_commit(bar_m2e);
            mma_px(T_DW(i), d, zprev, 2048, 144, acc);                            // wgrad_i main rows 0..127
            dbg();
            mma_px(T_PB(i), zprev, d + 16 * 2048, 2048, 16, acc);                 // wgrad_i rows 128,129 (transposed)
            dbg();
          } else {
            if constexpr (DX) mma_dx(t_addr(dbuf(0)));                            // 9 x 8 cycles: ahead of both commits
            if (more) {                                                           // next tile's input layer first:
              mma_input(a_txn);                                                   // its epilogue does not wait for
              dbg();
              tc::umma_commit(bar_m2e);                                           // this tile's input-layer wgrad
              mma_px(T_GIN, t_addr(dbuf(0)), a_tx, zero_a - a_tx, 16, acc);
              dbg();
            } else {
              mma_px(T_GIN, t_addr(dbuf(0)), a_tx, zero_a - a_tx, 16, acc);
              tc::umma_commit(bar_m2e);
            }
          }
          AWB_TR();
        }
      }
    }
  } else {
    // =========================================================== epilogue warps (12: 3 column groups x 4 lane quadrants)
    const int q = warp & 3, cg = warp >> 2;       // TMEM lanes [32q, 32q+32), stored chunks [6cg, 6cg + nch)
    const int row = q * 32 + lane;
    const uint32_t tlane = tbase + ((uint32_t)(q * 32) << 16);
    const int ch0 = 6 * cg;
    // The body is instantiated twice: for the column group that owns chunk 16 (5 stored chunks; columns 128..135 =
    // (z128, z129, x, y, [t,] 1, 0..), the corner sums) and for the other two (6 chunks) -- `last` and `nch` are
    // compile-time inside, so eight of the twelve warps carry none of the special cases' predicates.
    auto epilogue_body = [&](auto last_c) {
    constexpr bool last = decltype(last_c)::value;
    constexpr int nch = last ? 5 : 6;             // 6 + 6 + 5 = 17 stored chunks
    uint32_t ph = 0;
    float s_loss = 0.f, s_bo = 0.f, s_so0 = 0.f, s_so1 = 0.f, s_so2 = 0.f;   // cg 0: per-thread scalar sums
    float accC[L + 1];                            // cg 2: corner sums, lane-distributed (value = lane & 15)
#pragma unroll
    for (int i = 0; i <= L; i++) accC[i] = 0.f;
    const LossCoef ls = p.loss[o];
    // loss scale: host-chosen power of two, or (upstream-gradient mode) derived from the device-side max |dlogits|,
    // or (weighted loss) from max |w coef| over the kept pixels
    float S = p.scale[o];
    if (p.amax) { const float am = p.amax[o]; S = (am > 0.f && isfinite(am)) ? exp2f(rintf(log2f(64.f / am))) : 1.f; }
    LossPix lp = {};
    if constexpr (WL) {
      lp = p.pix[o];
      const float am = p.wamax[o] * p.coef_max[o];
      S = (am > 0.f && isfinite(am)) ? exp2f(rintf(log2f(64.f / am))) : 1.f;
    }
    constexpr bool has_dx = DX;
    float adx0 = 0.f, adx1 = 0.f, adx2 = 0.f;     // last group: d loss / d (x, y, t) of this row (scaled by S)
    // the input-layer part of it comes from the tensor pipe one round trip later: the row's sums and pixel wait for it
    float pdx0 = 0.f, pdx1 = 0.f, pdx2 = 0.f;
    int64_t pn = -1;
    auto flush_dx = [&]() {        // last group, after a wait on bar_m2e that covers the tile's DXIN contraction
      float g[4];
      tc::tmem_ld4(tlane + T_DX, g);
      tc::tmem_ld_wait();
      if (pn >= 0) {
        const float inv = 1.f / S;
        *reinterpret_cast<float4*>(p.dX + ((int64_t)o * p.N + pn) * 4) =
            make_float4((pdx0 + g[0]) * inv, (pdx1 + g[1]) * inv, C > 2 ? (pdx2 + g[2]) * inv : 0.f, 0.f);
      }
    };
    float v[48];
    const float* w = wo + 48 * cg;

    // accumulator columns [48cg, 48cg + 8nch) of this thread's row
    auto load_acc = [&](uint32_t taddr) {
      const uint32_t a = taddr + 48 * cg;
      tc::tmem_ld16(a, v); tc::tmem_ld16(a + 16, v + 16);
      if (last) tc::tmem_ld8(a + 32, v + 32); else tc::tmem_ld16(a + 32, v + 32);
      tc::tmem_ld_wait();
    };
    // arrive once per warp: every lane orders its generic-proxy stores and tcgen05.ld before the sync
    auto stage_done = [&]() {
      tc::fence_async_smem();
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(bar_e2m);
    };
    auto write_tx = [&](int buf, float a0, float a1, float a2) {
      if (cg == 0) st16(stx + buf * TX_B + row * 16, pack2(a0, a1), pack2(C > 2 ? a2 : 1.f, C > 2 ? 1.f : 0.f), 0u, 0u);
    };
    // coordinates / target of a tile (rows past N replicate the last pixel and carry no loss)
    float x0n = 0.f, x1n = 0.f, x2n = 0.f, tgtn = 0.f, wgtn = 1.f;
    bool liven = false;
    // Pixel position (frame, row, column) of this thread's row in the next tile to fetch, advanced tile by tile by
    // the decomposed tile stride: no integer divisions inside the tile loop.
    const uint32_t gW = (uint32_t)p.g.W, gH = (uint32_t)p.g.H, hw = gH * gW;
    uint32_t pb, pi, pj, db, di, dj;
    {
      const uint32_t n0 = p.g.row0 + blockIdx.x * 128u + (uint32_t)row, d = gridDim.x * 128u;   // global row
      pb = n0 / hw; uint32_t r = n0 - pb * hw; pi = r / gW; pj = r - pi * gW;
      db = d / hw; r = d - db * hw; di = r / gW; dj = r - di * gW;
    }
    const float sx = gW > 1 ? 1.0f / (float)(gW - 1) : 0.f, sy = gH > 1 ? 1.0f / (float)(gH - 1) : 0.f;   // lin01's steps
    auto lin = [](uint32_t i, uint32_t n, float step) {      // == lin01(i, n), bit for bit
      return n <= 1 ? 0.f : (i < n / 2 ? (float)i * step : 1.0f - (float)(n - 1 - i) * step);
    };
    auto fetch_tile = [&](int tile) {
      const int64_t n = (int64_t)tile * 128 + row;
      liven = n < p.N;
      if (p.X) {
        const uint32_t nn = (uint32_t)(liven ? n : p.N - 1);
        const float4 xv = *reinterpret_cast<const float4*>(p.X + ((int64_t)o * p.N + nn) * 4);
        x0n = xv.x; x1n = xv.y; x2n = C > 2 ? xv.z : 0.f;
      } else if (liven && p.g.mode == AWB_GRID_LINSPACE) {
        x2n = C > 2 ? p.g.t0 + (float)pb * p.g.t_step : 0.f;
        x0n = lin(pj, gW, sx); x1n = lin(pi, gH, sy);
      } else {      // padding rows of the last tile replicate the last pixel; explicit / index grids
        row_coords(p.g, (uint32_t)(liven ? n : p.N - 1), C, x0n, x1n, x2n);
      }
      pj += dj; if (pj >= gW) { pj -= gW; pi += 1; }
      pi += di; if (pi >= gH) { pi -= gH; pb += 1; }
      pb += db;
      tgtn = 0.f;
      if (fit && liven) tgtn = p.target[(int64_t)o * p.N + n];
      if constexpr (WL) wgtn = (liven && lp.weight) ? lp.weight[n] : 1.f;
    };
    auto chunk16_f32 = [&](const uint8_t* tile, float* c6) {   // columns 128..133 of a stored tile row
      const uint4 cz = *reinterpret_cast<const uint4*>(tile + 16 * 2048 + row * 16);
      c6[0] = half_lo(cz.x); c6[1] = half_hi(cz.x); c6[2] = half_lo(cz.y); c6[3] = half_hi(cz.y); c6[4] = half_lo(cz.z); c6[5] = half_hi(cz.z);
    };

    if (trace && warp == 0 && lane == 0) trace[121] = clock64();    // setup done
    fetch_tile(blockIdx.x);
    write_tx(0, x0n, x1n, x2n);
    stage_done();
    tc::mbar_wait(bar_w, 0);     // wo (read with plain loads below) has landed
    if (trace && warp == 0 && lane == 0) trace[122] = clock64();    // weights landed: tile loop starts

    for (int it = 0; it < n_my; it++) {
      const int tile = blockIdx.x + it * gridDim.x;
      const int64_t n = (int64_t)tile * 128 + row;
      const bool live = liven;
      const float x0 = x0n, x1 = x1n, x2 = x2n, tgt = tgtn, wgt = wgtn;
      const bool more = it + 1 < n_my;
      // aug values of chunk 16 columns 130..135: (x, y, [t,] 1, 0..)
      const uint32_t ax01 = pack2(x0, x1), ax2o = pack2(C > 2 ? x2 : 1.f, C > 2 ? 1.f : 0.f);

      // ---- stages 1..L: hidden forward epilogues (ACC -> relu -> ZT[s-1])
#pragma unroll
      for (int s = 1; s <= L; s++) {
        tc::mbar_wait(bar_m2e, ph); ph ^= 1;
        tc::fence_after_sync();
        AWB_TR();
        load_acc(tlane + T_ACC);
        AWB_TR();
        uint8_t* dst = tile_ptr(s - 1) + ch0 * 2048 + row * 16;
#pragma unroll
        for (int i = 0; i < 6; i++) {
          if (i < nch) {
            uint32_t w0 = pack2_relu(v[8 * i], v[8 * i + 1]), w1 = pack2_relu(v[8 * i + 2], v[8 * i + 3]);
            uint32_t w2 = pack2_relu(v[8 * i + 4], v[8 * i + 5]), w3 = pack2_relu(v[8 * i + 6], v[8 * i + 7]);
            if (last && i == 4) { w1 = ax01; w2 = ax2o; w3 = 0u; }
            st16(dst + i * 2048, w0, w1, w2, w3);
          }
        }
        AWB_TR();
        stage_done();
        AWB_TR();
      }

      // ---- stage L+1: last hidden activation, output layer, loss, delta_L
      tc::mbar_wait(bar_m2e, ph); ph ^= 1;
      tc::fence_after_sync();
      AWB_TR();
      load_acc(tlane + T_ACC);
      AWB_TR();
      {
        const int nz = last ? 34 : 48;                    // real z columns of this group
        float d4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < 48; j++) {
          if (j < nz) d4[j & 3] = fmaf(fmaxf(v[j], 0.f), w[j], d4[j & 3]);
        }
        float dot = (d4[0] + d4[1]) + (d4[2] + d4[3]);
        if (last) {
          dot = fmaf(x0, wo[H_], dot); dot = fmaf(x1, wo[H_ + 1], dot);
          if (C > 2) dot = fmaf(x2, wo[H_ + 2], dot);
          dot += wo[H_ + C];
        }
        xchg[cg * 128 + row] = dot;
      }
      // z_L as packed fp16 pairs: operand tile of the output-layer wgrad, then turned into the relu mask
      uint32_t zp[24];
#pragma unroll
      for (int k = 0; k < 24; k++) zp[k] = pack2_relu(v[2 * k], v[2 * k + 1]);
      const float zL128 = last ? half_lo(zp[16]) : 0.f, zL129 = last ? half_hi(zp[16]) : 0.f;
      if (fit) {
        uint8_t* zl = tile_ptr(L) + ch0 * 2048 + row * 16;
#pragma unroll
        for (int i = 0; i < 6; i++) {
          if (i < nch) {
            if (last && i == 4) st16(zl + i * 2048, zp[16], 0u, 0u, 0u);
            else st16(zl + i * 2048, zp[4 * i], zp[4 * i + 1], zp[4 * i + 2], zp[4 * i + 3]);
          }
        }
#pragma unroll
        for (int k = 0; k < 24; k++) zp[k] = gt0_mask2(zp[k]);
      }
      AWB_TR();
      asm volatile("bar.sync %0, 96;" ::"r"(1 + q) : "memory");   // the three warps that share these 32 rows
      const float y = (xchg[row] + xchg[128 + row]) + xchg[256 + row];
      AWB_TR();
      if (!fit) {
        if (cg == 0 && live && p.logits) p.logits[(int64_t)o * p.N + n] = y;
        if (more) { fetch_tile(tile + gridDim.x); write_tx((it + 1) & 1, x0n, x1n, x2n); }
        stage_done();
        continue;
      }
      float dys = 0.f, lossv = 0.f;
      if (live) {
        const bool fg = ls.cls_rule == AWB_CLS_UNARY_LT_HALF ? (tgt < 0.5f) : (tgt != 1.0f);
        const float coef = WL ? (fg ? ls.coef_fg : ls.coef_bg) * wgt : (fg ? ls.coef_fg : ls.coef_bg);
        const float sg = __fdividef(1.f, 1.f + __expf(-y));
        float l, dl;
        if (ls.kind == AWB_LOSS_SE_SIGMOID) { float d = tgt - sg; l = d * d; dl = -2.f * d * sg * (1.f - sg); }
        else if (ls.kind == AWB_LOSS_UPSTREAM) { l = 0.f; dl = tgt; }       // `target` holds d loss / d logits (autograd)
        else { l = bce_logits(y, tgt); dl = sg - tgt; }
        dys = coef * dl * S;
        lossv = coef * l;
        if (WL && !loss_keep(lp, tgt)) { dys = 0.f; lossv = 0.f; }      // select: a NaN there cannot leak in
      }
      // delta_L = dy * w_o .* (z_L > 0) on packed fp16 pairs
      float dL128 = 0.f, dL129 = 0.f;
      {
        uint8_t* dl = dbuf(L) + ch0 * 2048 + row * 16;
        const uint32_t dys2 = pack2(dys, dys);
        const __half2 dh = *reinterpret_cast<const __half2*>(&dys2);
        auto dmul = [&](uint32_t wq, uint32_t m) {
          __half2 r = __hmul2(dh, *reinterpret_cast<const __half2*>(&wq));
          return *reinterpret_cast<uint32_t*>(&r) & m;
        };
#pragma unroll
        for (int i = 0; i < 6; i++) {
          if (i < nch) {
            const uint4 wq = *reinterpret_cast<const uint4*>(wo16 + (ch0 + i) * 16);
            uint32_t w0 = dmul(wq.x, zp[4 * i]), w1 = dmul(wq.y, zp[4 * i + 1]), w2 = dmul(wq.z, zp[4 * i + 2]), w3 = dmul(wq.w, zp[4 * i + 3]);
            if (last && i == 4) {
              dL128 = half_lo(w0); dL129 = half_hi(w0);
              w1 = pack2(dys, 0.f); w2 = 0u; w3 = 0u;
            }
            st16(dl + i * 2048, w0, w1, w2, w3);
          }
        }
      }
      AWB_TR();
      stage_done();
      AWB_TR();
      // ---- shadow of dgrad_L: everything that is not an operand of the next contraction
      if (cg == 0) {
        if (p.logits && live) p.logits[(int64_t)o * p.N + n] = y;
        s_loss += lossv; s_bo += dys;
        s_so0 += dys * x0; s_so1 += dys * x1;
        if (C > 2) s_so2 += dys * x2;
      } else if (last) {
        if (has_dx && it > 0) flush_dx();      // previous tile's coordinate gradient (its contraction finished rounds ago)
        // corner of dW_L: delta_L[128..129] x ZT[L-1][128..133], and d w_o[128], [129]
        float c6[6], cv[16];
        chunk16_f32(tile_ptr(L - 1), c6);
#pragma unroll
        for (int b = 0; b < 6; b++) { cv[b] = dL128 * c6[b]; cv[6 + b] = dL129 * c6[b]; }
        cv[12] = zL128 * dys; cv[13] = zL129 * dys; cv[14] = 0.f; cv[15] = 0.f;
        accC[L] += warp_reduce_scatter16(cv, lane);
        if (has_dx) { adx0 = dys * wo[H_]; adx1 = dys * wo[H_ + 1]; adx2 = C > 2 ? dys * wo[H_ + 2] : 0.f; }   // out.skp
      }
      if (more) fetch_tile(tile + gridDim.x);     // next tile's coordinates and target (load latency hidden)

      // ---- stages L+2 .. 2L+1: backward hidden epilogues: ACC = dZA_{i-1} -> delta_{i-1}
#pragma unroll
      for (int i = L; i >= 1; i--) {
        // relu mask of z_{i-1} from the stored activations, before the wait
        uint32_t mk[24];
        {
          const uint8_t* zsrc = tile_ptr(i - 1) + ch0 * 2048 + row * 16;
#pragma unroll
          for (int c = 0; c < 6; c++) {
            if (c < nch) {
              const uint4 u = *reinterpret_cast<const uint4*>(zsrc + c * 2048);
              mk[4 * c] = gt0_mask2(u.x); mk[4 * c + 1] = gt0_mask2(u.y); mk[4 * c + 2] = gt0_mask2(u.z); mk[4 * c + 3] = gt0_mask2(u.w);
            }
          }
        }
        tc::mbar_wait(bar_m2e, ph); ph ^= 1;
        tc::fence_after_sync();
        AWB_TR();
        load_acc(tlane + T_ACC);
        if (last && has_dx) { adx0 += v[34]; adx1 += v[35]; if (C > 2) adx2 += v[36]; }   // skip-connection columns of dZA
        uint8_t* dst = dbuf(i - 1) + ch0 * 2048 + row * 16;
        float d128 = 0.f, d129 = 0.f;
#pragma unroll
        for (int c = 0; c < 6; c++) {
          if (c < nch) {
            uint32_t w0 = pack2(v[8 * c], v[8 * c + 1]) & mk[4 * c], w1 = pack2(v[8 * c + 2], v[8 * c + 3]) & mk[4 * c + 1];
            uint32_t w2 = pack2(v[8 * c + 4], v[8 * c + 5]) & mk[4 * c + 2], w3 = pack2(v[8 * c + 6], v[8 * c + 7]) & mk[4 * c + 3];
            if (last && c == 4) {
              w1 = 0u; w2 = 0u; w3 = 0u;
              d128 = (mk[16] & 0xFFFFu) ? v[32] : 0.f;
              d129 = (mk[16] >> 16) ? v[33] : 0.f;
            }
            st16(dst + c * 2048, w0, w1, w2, w3);
          }
        }
        if (i == 1 && more) write_tx((it + 1) & 1, x0n, x1n, x2n);   // next tile's input operand rides this round trip
        stage_done();
        AWB_TR();
        if (last) {
          float cv[16];
          if (i - 1 >= 1) {   // corner of dW_{i-1}
            float c6[6];
            chunk16_f32(tile_ptr(i - 2), c6);
#pragma unroll
            for (int b = 0; b < 6; b++) { cv[b] = d128 * c6[b]; cv[6 + b] = d129 * c6[b]; }
            cv[12] = 0.f; cv[13] = 0.f; cv[14] = 0.f; cv[15] = 0.f;
          } else {            // corner of the input layer: delta_0[128..129] x (x, y, t, 1)
            cv[0] = d128 * x0; cv[1] = d128 * x1; cv[2] = d128 * x2; cv[3] = d128;
            cv[4] = d129 * x0; cv[5] = d129 * x1; cv[6] = d129 * x2; cv[7] = d129;
#pragma unroll
            for (int b = 8; b < 16; b++) cv[b] = 0.f;
          }
          accC[i - 1] += warp_reduce_scatter16(cv, lane);
        }
        if (i == 1 && has_dx && last) { pdx0 = adx0; pdx1 = adx1; pdx2 = adx2; pn = live ? n : -1; }
      }
    }

    // the last commit (input-layer wgrad of the last tile / last forward stage) closes the pipeline
    tc::mbar_wait(bar_m2e, ph); ph ^= 1;
    tc::fence_after_sync();
    AWB_TR();
    if (has_dx && fit && last && n_my > 0) flush_dx();              // the last tile's coordinate gradient
    if (trace && warp == 0 && lane == 0) trace[123] = clock64();    // tile loop done

    // =========================================================== per-CTA partial write-out
    if (fit) {
      const float inv = 1.f / S;
      float* out = p.part + (int64_t)blockIdx.x * p.sSplit + (int64_t)o * p.G;
      const int et = warp * 32 + lane;                    // 0..383
      // scalar / corner sums: fixed-order reduction through shared memory (scratch: the dead weight image)
      float* redS = reinterpret_cast<float*>(simg);       // [5][128]   per-row scalars of column group 0
      float* redC = redS + 5 * 128;                       // [L+1][4][16] lane-distributed corner sums of group 2
      if (cg == 0) {
        redS[row] = s_loss; redS[128 + row] = s_bo; redS[256 + row] = s_so0; redS[384 + row] = s_so1; redS[512 + row] = s_so2;
      } else if (last && lane < 16) {
#pragma unroll
        for (int i = 0; i <= L; i++) redC[(i * 4 + q) * 16 + lane] = accC[i];
      }
      // dW_i main rows: TMEM -> registers -> staging tile [128][136] fp32 (the dead operand tiles)
      float* stage = reinterpret_cast<float*>(tiles);     // [L][128][136]
#pragma unroll
      for (int i = 1; i <= L; i++) {
        load_acc(tlane + T_DW(i));
        float* dst = stage + (i - 1) * 128 * LD_ + row * LD_ + 48 * cg;
        const int nv = 2 * nch;
#pragma unroll
        for (int j = 0; j < 12; j++)
          if (j < nv) *reinterpret_cast<float4*>(dst + 4 * j) = make_float4(v[4 * j] * inv, v[4 * j + 1] * inv, v[4 * j + 2] * inv, v[4 * j + 3] * inv);
        if (cg == 0) {
          float pb[8];
          tc::tmem_ld8(tlane + T_PB(i), pb);
          tc::tmem_ld_wait();
          float* l = out + p.aug_layer + (int64_t)(i - 1) * H_ * LD_;
          l[(int64_t)128 * LD_ + row] = pb[0] * inv;
          l[(int64_t)129 * LD_ + row] = pb[1] * inv;
        }
      }
      if (cg == 0) {
        float g8[8];
        tc::tmem_ld8(tlane + T_GIN, g8);
        tc::tmem_ld_wait();
        float* gi = out + p.aug_in + row * 4;
        float4 gv;
        gv.x = g8[0] * inv; gv.y = g8[1] * inv;
        if (C > 2) { gv.z = g8[2] * inv; gv.w = g8[3] * inv; } else { gv.z = 0.f; gv.w = g8[2] * inv; }
        *reinterpret_cast<float4*>(gi) = gv;
        tc::tmem_ld8(tlane + T_GO, g8);
        tc::tmem_ld_wait();
        out[p.aug_out + row] = g8[2] * inv;
      }
      tc::fence_async_smem();
      asm volatile("bar.sync 5, %0;" ::"n"(NEW * 32) : "memory");
      if (et == 0) {   // TMA bulk stores of the staged main rows (contiguous [128][136] fp32 per layer)
#pragma unroll
        for (int i = 1; i <= L; i++) {
          float* gdst = out + p.aug_layer + (int64_t)(i - 1) * H_ * LD_;
          asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
                       "r"(tc::smem_u32(stage + (i - 1) * 128 * LD_)), "r"((uint32_t)(128 * LD_ * 4)) : "memory");
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
      if (warp >= 1 && warp <= 5) {   // scalars: lanes stride the 128 rows, fixed order
        const int i = warp - 1;
        float a = 0.f;
#pragma unroll
        for (int k = 0; k < 4; k++) a += redS[i * 128 + lane + 32 * k];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
        if (lane == 0) {
          if (i == 0) p.lossp[blockIdx.x * p.O + o] = a;
          else if (i == 1) out[p.aug_out + H_ + C] = a * inv;             // d b_o
          else if (i - 2 < C) out[p.aug_out + H_ + (i - 2)] = a * inv;    // d s_o
        }
      } else if (warp >= 6 && et - 192 < (L + 1) * 16) {   // corners: four quadrant partials each
        const int li = (et - 192) >> 4, sl = (et - 192) & 15;
        float a = 0.f;
#pragma unroll
        for (int qq = 0; qq < 4; qq++) a += redC[(li * 4 + qq) * 16 + sl];
        a *= inv;
        if (li == 0) {
          // (x, y, t, 1) order of the accumulators -> (w_x, w_y, w_t, bias) slots; C == 2 keeps slot 2 zero
          if (sl < 8) out[p.aug_in + (128 + (sl >> 2)) * 4 + (sl & 3)] = (C == 2 && (sl & 3) == 2) ? 0.f : a;
        } else {
          if (sl < 12) {
            const int r = sl / 6, b = sl % 6;
            if (b < 3 + C) out[p.aug_layer + (int64_t)(li - 1) * H_ * LD_ + (int64_t)(128 + r) * LD_ + 128 + b] = a;
          } else if (li == L && sl < 14) {
            out[p.aug_out + 128 + (sl - 12)] = a;
          }
        }
      }
      // the CTA may exit once the bulk stores have read their shared-memory source; kernel completion covers the writes
      if (et == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    if (trace && warp == 0 && lane == 0) {                     // write-out done
      trace[124] = clock64();
      unsigned long long ns;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
      trace[126] = ns;
    }
    };   // epilogue_body
    if (cg == NCG - 1) epilogue_body(std::true_type{});
    else epilogue_body(std::false_type{});
  }
  tc::fence_before_sync();
  __syncthreads();
  if (issuer_warp) tc::tmem_dealloc<512>(tbase);
#undef AWB_TR
}

// ======================================================================= host launcher
int tc_supported(const awb_prior* h) {
  return (h->desc.kind == AWB_KIND_ICNN || h->desc.kind == AWB_KIND_FLOW_ICNN || h->desc.kind == AWB_KIND_DIFFEO_ICNN) && h->lay.h == H_ &&
         (h->lay.L == 1 || h->lay.L == 2) && h->lay.ld == LD_;
}

int tc_map_elems(int L) { return (L * W_B + WIN_B) / 2 + 2 * NPAD; }

// image element index -> arena index (or -1)
void tc_build_map_host(const Layout& Ly, int32_t* map) {
  const int L = Ly.L, C = Ly.C;
  const int n_half = (L * W_B + WIN_B) / 2;
  for (int i = 0; i < n_half + 2 * NPAD; i++) map[i] = -1;
  // arena order (state_dict): input.weight [h][C], input.bias [h], {ln.weight [h][h], ln.bias [h], skp.weight [h][C]} x L,
  // out.ln.weight [h], out.ln.bias, out.skp.weight [C]
  int64_t a = Ly.off_icnn;
  auto w_elem = [&](int l, int j, int k) { return l * (W_B / 2) + (k / 8) * (NPAD * 8) + j * 8 + (k % 8); };
  auto win_elem = [&](int j, int k) { return L * (W_B / 2) + j * 8 + k; };   // one stored K chunk (k < 8)
  for (int j = 0; j < H_; j++) for (int c = 0; c < C; c++) map[win_elem(j, c)] = (int32_t)a++;
  for (int j = 0; j < H_; j++) map[win_elem(j, C)] = (int32_t)a++;
  for (int l = 0; l < L; l++) {
    for (int j = 0; j < H_; j++) for (int k = 0; k < H_; k++) map[w_elem(l, j, k)] = (int32_t)a++;
    for (int j = 0; j < H_; j++) map[w_elem(l, j, H_ + C)] = (int32_t)a++;
    for (int j = 0; j < H_; j++) for (int c = 0; c < C; c++) map[w_elem(l, j, H_ + c)] = (int32_t)a++;
  }
  for (int k = 0; k < H_; k++) map[n_half + k] = (int32_t)a++;
  map[n_half + H_ + C] = (int32_t)a++;
  for (int c = 0; c < C; c++) map[n_half + H_ + c] = (int32_t)a++;
  for (int k = 0; k < NPAD; k++) map[n_half + NPAD + k] = map[n_half + k];   // fp16 copy of the output vector
}

// augmented index -> fp16 element index of the weight image (hidden layers and input layer; the output vector
// is handled by its own fp32 + fp16 slots, see k_reduce_opt_aug)
void tc_build_aug2img_host(const Layout& Ly, int32_t* a2i) {
  const int L = Ly.L, C = Ly.C;
  for (int64_t i = 0; i < Ly.G; i++) a2i[i] = -1;
  for (int j = 0; j < H_; j++) {
    for (int c = 0; c < C; c++) a2i[Ly.aug_in + j * 4 + c] = L * (W_B / 2) + j * 8 + c;
    a2i[Ly.aug_in + j * 4 + 3] = L * (W_B / 2) + j * 8 + C;
  }
  for (int l = 0; l < L; l++)
    for (int j = 0; j < H_; j++)
      for (int k = 0; k < H_ + C + 1; k++)
        a2i[Ly.aug_layer + (int64_t)l * H_ * LD_ + (int64_t)j * LD_ + k] = l * (W_B / 2) + (k / 8) * (NPAD * 8) + j * 8 + (k % 8);
}

int64_t tc_vec_offset_bytes(int L) { return (int64_t)L * W_B + WIN_B; }

static unsigned long long* g_trace_dev = nullptr;   // debug timeline buffer (AWB_TC_TRACE=1), [grid][TRACE_N]
static int g_trace_ctas = 0;

int tc_trace_read(unsigned long long* host, int max_ctas) {
  if (!g_trace_dev) return 0;
  int n = g_trace_ctas < max_ctas ? g_trace_ctas : max_ctas;
  cudaDeviceSynchronize();
  cudaMemcpy(host, g_trace_dev, sizeof(unsigned long long) * TRACE_N * n, cudaMemcpyDeviceToHost);
  return n;
}

int tc_fit_forward_backward(const awb_prior* h, const float* params, const awb_grid_spec* g, const float* target,
                            const awb_loss_spec* loss, float* logits, int mode, const Workspace& ws, int* n_splits_out,
                            cudaStream_t st, bool reuse_packed, const float* Xrows, float* dXrows, const float* amax,
                            const float* wamax) {
  const Layout& Ly = h->lay;
  const int O = h->desc.n_objects, L = Ly.L, C = Ly.C;
  const int64_t N = ws.N;
  if (!tc_supported(h)) { set_error("precision f16 supports ICNN / flow+ICNN priors with h=130, L in {1,2}"); return AWB_ERR_UNSUPPORTED; }
  const int n_tiles = (int)((N + 127) / 128);
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
  // One wave: the O objects share the SMs (sms / O persistent CTAs each).  Compared with sms CTAs per object in O
  // waves this keeps the number of gradient partials (and their L2 footprint, and the optimizer kernel's reads) at
  // one per SM in total, removes the tile quantisation (2400 tiles / 37 CTAs = 64.9 -> 65 instead of 16.2 -> 17 per
  // frame at O = 4) and pays the per-CTA weight load and partial write-out once per SM instead of once per SM and object.
  const int per_obj = sms / O > 0 ? sms / O : 1;
  const int grid = n_tiles < per_obj ? n_tiles : per_obj;
  if (grid > kMaxSplits) { set_error("internal: grid exceeds split capacity"); return AWB_ERR_INVALID; }
  const int64_t img_stride = tc_image_bytes(L);
  const int n_elems = tc_map_elems(L);
  if (!reuse_packed)   // otherwise the optimizer kernel of the previous fit step left the image up to date
    AWB_LAUNCH(PK_PACK, st, k_pack_tc<<<dim3((n_elems + 255) / 256, O), 256, 0, st>>>(params, (uint8_t*)ws.tc, h->d_tcmap, n_elems,
                                                                                      L, Ly.P, img_stride));
  TcP p = {};
  p.g.mode = g->mode; p.g.B = g->B; p.g.H = g->H; p.g.W = g->W; p.g.C = C; p.g.t0 = g->t0; p.g.t_step = g->t_step; p.g.grid = g->grid;
  p.g.row0 = (uint32_t)ws.row0;
  p.img = (const uint8_t*)ws.tc; p.img_stride = img_stride;
  p.target = target;
  for (int o = 0; o < O && o < 16; o++) {
    if (loss) {
      p.loss[o] = loss_coef(loss[o]);
      float mx = fmaxf(fabsf(loss[o].coef_fg), fabsf(loss[o].coef_bg));
      p.scale[o] = mx > 0.f ? exp2f(rintf(log2f(64.f / mx))) : 1.f;   // keeps fp16 deltas in range (loss scaling)
      p.pix[o] = loss_pix(loss[o]);
      p.coef_max[o] = mx;
    } else {
      p.scale[o] = 1.f;
    }
  }
  p.part = ws.part; p.sSplit = (int64_t)O * Ly.G; p.G = Ly.G; p.aug_in = Ly.aug_in; p.aug_layer = Ly.aug_layer; p.aug_out = Ly.aug_out;
  p.lossp = ws.lossp; p.O = O; p.logits = logits; p.N = N; p.n_tiles = n_tiles; p.mode = mode;
  p.X = Xrows; p.dX = dXrows; p.amax = amax; p.wamax = wamax;
  p.trace = nullptr;
  if (const char* tr = getenv("AWB_TC_TRACE")) {
    p.trace_serial = atoi(tr) == 2;
    if (!g_trace_dev) cudaMalloc(&g_trace_dev, sizeof(unsigned long long) * TRACE_N * kMaxSplits * 16);
    if (g_trace_dev) { cudaMemsetAsync(g_trace_dev, 0, sizeof(unsigned long long) * TRACE_N * grid * O, st); p.trace = g_trace_dev; g_trace_ctas = grid * O; }
  }
  const size_t smem = smem_bytes(L);
  dim3 gd(grid, O);
#define AWB_TC_LAUNCH3(LL, CC, FF, DD, WW)                                                                             \
  do {                                                                                                             \
    AWB_CUDA(cudaFuncSetAttribute(k_icnn_fit_tc<LL, CC, FF, DD, WW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    AWB_LAUNCH(PK_TC_FUSED, st, AWB_CUDA(launch_ex(k_icnn_fit_tc<LL, CC, FF, DD, WW>, gd, dim3(NTHREADS), smem, st, true, p))); \
  } while (0)
#define AWB_TC_LAUNCH(LL, CC)                                              \
  do {                                                                     \
    if (mode == 0) AWB_TC_LAUNCH3(LL, CC, false, false, false);            \
    else if (wamax && dXrows) AWB_TC_LAUNCH3(LL, CC, true, true, true);    \
    else if (wamax) AWB_TC_LAUNCH3(LL, CC, true, false, true);             \
    else if (dXrows) AWB_TC_LAUNCH3(LL, CC, true, true, false);            \
    else AWB_TC_LAUNCH3(LL, CC, true, false, false);                       \
  } while (0)
  if (L == 1 && C == 2) AWB_TC_LAUNCH(1, 2);
  else if (L == 1 && C == 3) AWB_TC_LAUNCH(1, 3);
  else if (L == 2 && C == 2) AWB_TC_LAUNCH(2, 2);
  else AWB_TC_LAUNCH(2, 3);
#undef AWB_TC_LAUNCH
#undef AWB_TC_LAUNCH3
  AWB_CUDA(cudaGetLastError());
  if (n_splits_out) *n_splits_out = grid;
  return AWB_OK;
}

}  // namespace awb
