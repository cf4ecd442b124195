// Internal declarations shared by the translation units of libawb.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/awb.h"

namespace awb {

constexpr int kMaxSplits = 148;  // pixel ranges for cross-pixel reductions = one per SM
constexpr int kMaxObjects = 64;

// Per-object layout of the parameter arena (state_dict order) and of the "augmented"
// weight space the kernels consume.
//
// Augmented formulation (DESIGN.md): every hidden activation row is stored as
//   ZA[n] = [ z (h) | x (C) | 1 | 0-pad ]           (ld = round_up(h+C+1, 8) floats)
// and every SkipBlock as one matrix  Waug[h][ld] = [ ln.weight | skp.weight | ln.bias | 0 ],
// so that  z_{i+1} = relu(ZA_i * Waug^T),  dZA_i = delta * Waug  (its x-columns are the
// coordinate gradient) and  dWaug = delta^T * ZA_i  (dW, dS, db in one contraction).
struct Layout {
  int C, h, L, F, m, ld;
  int64_t P;         // trainable parameters per object
  int64_t off_icnn;  // arena offset of input.weight
  int64_t P_icnn;
  int64_t off_flow;  // arena offset of flows.0.s.net.0.weight
  int64_t P_flow;    // F * per_flow
  int64_t per_flow;  // 2*(m*C + m + C*m + C) + 2*C
  int64_t off_lin;   // arena offset of linear.weight, linear.bias
  int64_t n_lin;     // their size: 2C (grouped 1x1 conv of PathConnectedNet) or C*C + C (nn.Linear of ConvexDiffeomorphismNet)
  // augmented space
  int64_t G;         // 4*h + L*h*ld + ld
  int64_t aug_in;    // [h][4]: (w_x, w_y, w_t, bias)
  int64_t aug_layer; // + i*h*ld, i < L
  int64_t aug_out;   // [ld]: (w_o | s_o | b_o | 0)
};

struct OptScal {  // per object, device resident
  double lr[AWB_MAX_GROUPS];
  double best;
  int32_t step;
  int32_t num_bad;
  int32_t nonfinite;
  int32_t pad;
  float last_loss;
  float pad2;
  int32_t group_start[AWB_MAX_GROUPS];   // steps this group sat out (not in active_groups).  torch keeps a step counter per
                                         // parameter and does not advance it while the grad is None, so the group's own
                                         // count -- the one its bias correction uses -- is step - group_start[g]
};

struct FlowConsts {
  float nmin[4], nmax[4];
  float new_min, new_max;
  float out_scale;        // output_scale of the coupling MLPs (1 when unset)
  uint8_t masks[64 * 4];  // [F][C]
};

}  // namespace awb

struct awb_prior {
  awb_desc desc;
  awb::Layout lay;
  int32_t* d_map;     // [P_icnn] arena-local index -> augmented index
  uint8_t* d_clamp;   // [P] 1 where enforce_convexity clamps
  uint8_t* d_group;   // [P] optimizer group: 0 flow_net, 1 convex_net, 2 linear
  int32_t* d_tcmap;   // tensor path: weight-image element -> arena index (or -1), null when unsupported
  int32_t* d_imap;    // [G] augmented index -> arena-local ICNN index (or -1 for padding)
  int32_t* d_aug2img; // tensor path: [G] augmented index -> fp16 element of the weight image (or -1)
  awb::FlowConsts fc;
  bool fc_set;
  int flow_eval;      // RealNVP coupling MLPs: 0 auto, 1 unit loops, 2 segment tables (awb_prior_set_flow_eval)
  int device;
  // awb_prior_fit_host_frames: copy stream + staging-buffer events, created on first use
  cudaStream_t copy_stream;
  cudaEvent_t ev_ready[2], ev_free[2];
  bool stream_made;
};

namespace awb {

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
#define AWB_CUDA(expr)                                    \
  do {                                                    \
    cudaError_t _e = (expr);                              \
    if (_e != cudaSuccess) return awb::cuda_fail(_e, #expr); \
  } while (0)

inline int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }
inline int n_splits(int64_t n) {
  int64_t s = (n + 255) / 256;
  return (int)(s < kMaxSplits ? (s < 1 ? 1 : s) : kMaxSplits);
}
inline int64_t split_chunk(int64_t n) { return round_up((n + n_splits(n) - 1) / n_splits(n), 8); }

// Workspace carving (all regions 256-byte aligned).
struct Workspace {
  float* waug;    // [O][G]
  float* part;    // [S][O][G]
  float* lossp;   // [S][O]
  float* fpart;   // [S][O][P_flow + 2C]   (flow + linear gradient partials)
  float* X;       // [O][N][4]   deformed coordinates fed to the ICNN (x, y, t, 1)
  float* dX;      // [O][N][4]
  float* ZA;      // [O][L+1][N][ld]
  float* D;       // [O][2][N][ld]
  float* logits;  // [O][N]
  float* flowz;   // training, flow priors: saved coupling inputs.  RealNVP: [O][F][N][RW] (input + s, t outputs of every
                  // coupling, awb_flow.cu FlowSave); NormalizingFlow1D: [O][N][F*C]
  float* flowd;   // RealNVP backward, C = 3, pixel ranges too large for shared memory: [O][N][4] scratch
  float* flowtab; // RealNVP, C = 2: [O][F][2][132] segment tables of the coupling MLPs, rebuilt by every forward
  float* flowseg; // RealNVP, C = 2, training: [S][O][F][8][144] per-warp histogram sums of the segment backward
  void* tc;       // tensor-core path scratch
  float* ZT;      // second-order pass (awb_prior_grid_grad_backward): [L+1][N][ld] tangent rows, after everything else so
                  // that the training forward's layout is a prefix of this one
  int64_t bytes;
  // the pixel rows [row0, row0 + N) of the grid's batch this call works on: the whole batch (row0 = 0) for every entry
  // point but awb_prior_slice_grads.  Kernels index their scratch and the target by the local row and generate (or read)
  // coordinates at the global one.
  int64_t row0, N;
};
// Regions of workspace layout `layout` (AWB_WS_*, validated by the caller) for N pixel rows at base (null: sizes only).
// AWB_WS_DEFORMATION: flow buffers only (X, coupling records, dX, flow partials and scratch), no ICNN weights, partials
// or activation planes.  AWB_WS_SECOND_ORDER: the training layout plus the tangent rows ZT.
Workspace carve(const awb_prior* h, int64_t N, int layout, void* base);

// ---- per-kernel-class timing (CUDA events on the launch stream) and launch counting ----
enum { PK_PACK = 0, PK_INPUT, PK_GEMM_FWD, PK_OUT_LOSS, PK_GEMM_WGRAD, PK_GEMM_DGRAD, PK_IN_BWD, PK_OPT,
       PK_FLOW_FWD, PK_FLOW_BWD, PK_TC_FUSED, PK_MISC, PK_TAN_FWD, PK_TAN_OUT, PK_COUNT };
void prof_begin(int cls, cudaStream_t st);
void prof_end(int cls, cudaStream_t st);
#define AWB_LAUNCH(cls, st, ...)  \
  do {                            \
    awb::prof_begin(cls, st);     \
    __VA_ARGS__;                  \
    awb::prof_end(cls, st);       \
  } while (0)

// Launch with (optionally) programmatic stream serialization: the kernel may become resident while its predecessor in
// the stream drains.  Every kernel launched this way executes griddepcontrol.wait before it touches global memory
// and griddepcontrol.launch_dependents only after that wait, so completion stays transitive along the stream.
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_ex(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                             Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = (pdl && pdl_enabled()) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- launchers implemented in awb_simt.cu ----
struct GridDev {
  int mode, B, H, W, C;
  float t0, t_step;
  const float* grid;
  uint32_t row0;   // global index of local row 0 (Workspace::row0)
};
int simt_forward(const awb_prior* h, const float* params, const awb_grid_spec* g, float* logits_out,
                 float* deformed, bool training, const Workspace& ws, cudaStream_t st);
// loss != nullptr: fit mode (dy from loss); else dy = dlogits.
// dgrid (optional, flow priors): the flow backward also writes d / d grid, planar [B,C,H,W]
int simt_backward(const awb_prior* h, const float* params, const awb_grid_spec* g, const float* target,
                  const awb_loss_spec* loss, const float* dlogits, bool need_dx, const Workspace& ws,
                  cudaStream_t st, float* dgrid = nullptr);
// n_partials: number of ICNN gradient partials ([S][O][G]) the producer wrote (-1: n_splits(N)); the flow
// partials always come from flow_backward's n_splits(N) pixel ranges.
int simt_reduce_opt(const awb_prior* h, float* params, void* opt_state, const awb_opt_hyper* hy,
                    float* loss_out, const Workspace& ws, int64_t N, cudaStream_t st, int n_partials = -1);
// loss_slot (optional, single object): receives the sum of the loss partials (gradient row of awb_prior_slice_grads).
// n_partials = 0: no ICNN partials were written (flow-only backward), the ICNN entries of grads are exactly 0.
int simt_reduce_grads(const awb_prior* h, float* grads, const Workspace& ws, int64_t N, cudaStream_t st, int n_partials = -1,
                      float* loss_slot = nullptr);
// second-order pass of the coordinate gradient (single-object ICNN, after simt_forward(training) on ws, ws carved with
// tangent rows): d_dgrid [B,C,H,W] -> ydot [N] and the parameter-gradient partials that simt_reduce_grads sums
int simt_grid_grad_backward(const awb_prior* h, const awb_grid_spec* g, const float* dlogits, const float* d_dgrid,
                            float* ydot, const Workspace& ws, cudaStream_t st);
int absmax_per_object(const float* x, int64_t n, int O, float* out, cudaStream_t st);   // out[o] = max |x[o][:]|
int simt_dgrid(const awb_prior* h, const awb_grid_spec* g, float* dgrid, const Workspace& ws, cudaStream_t st);
// ws.dX[n] = (d_deformed[n][0..C), 0...): seeds the flow backward with a caller gradient on the deformed coordinates
int simt_seed_dX(const awb_prior* h, const float* d_deformed, const Workspace& ws, cudaStream_t st);
int optim_step(const awb_prior* h, float* params, const float* grads, void* opt_state,
               const awb_opt_hyper* hy, cudaStream_t st);
int clamp_only(const awb_prior* h, float* params, cudaStream_t st);
int plateau_step(const awb_prior* h, void* opt_state, const float* loss, int stride, const awb_opt_hyper* hy, cudaStream_t st);
// reduce [S][P] plain (state_dict order) gradient partials + [S] loss partials, then the optimizer step
// (partial s at partials + s * part_stride, its loss at lossp[s * loss_stride]; awb_prior_rows_opt_step: the loss is
// column P of each gradient row)
int reduce_opt_plain(const awb_prior* h, float* params, void* opt_state, const awb_opt_hyper* hy, float* loss_out,
                     const float* partials, int S, int64_t part_stride, const float* lossp, int64_t loss_stride,
                     cudaStream_t st);
// ---- star-shape prior, implemented in awb_star.cu
int star_n_ctas(int64_t n);
int star_run(const awb_prior* h, const float* params, const float* x, const float* target, int64_t n,
             const awb_loss_spec* loss, float* logits, float* part, float* lossp, bool fit, int* n_ctas, cudaStream_t st);
int opt_state_init(const awb_prior* h, void* opt_state, const double* lr, cudaStream_t st);
int opt_set_lr(const awb_prior* h, void* opt_state, const double* lr, cudaStream_t st);

// ---- tensor path (tcgen05), implemented in awb_tc_fit.cu ----
int tc_supported(const awb_prior* h);
int tc_image_bytes(int L);
int tc_map_elems(int L);
void tc_build_map_host(const Layout& Ly, int32_t* map);   // map has tc_map_elems(L) entries
void tc_build_aug2img_host(const Layout& Ly, int32_t* a2i);   // a2i has Ly.G entries
int64_t tc_vec_offset_bytes(int L);                       // byte offset of the fp32 output vector inside the image
// mode 0: forward only (logits), mode 1: forward + loss + backward partials (part / lossp, *n_splits_out CTAs)
int tc_fit_forward_backward(const awb_prior* h, const float* params, const awb_grid_spec* g, const float* target,
                            const awb_loss_spec* loss, float* logits, int mode, const Workspace& ws,
                            int* n_splits_out, cudaStream_t st, bool reuse_packed = false,
                            const float* Xrows = nullptr, float* dXrows = nullptr, const float* amax = nullptr);
int tc_trace_read(unsigned long long* host, int max_ctas);   // debug timeline (AWB_TC_TRACE=1): 256 stamps per CTA

// ---- flows, implemented in awb_flow.cu ----
int flow_forward(const awb_prior* h, const float* params, const awb_grid_spec* g, const Workspace& ws,
                 float* deformed, cudaStream_t st, bool use_linear = true);
int flow_inverse(const awb_prior* h, const float* params, const awb_grid_spec* g, float* out, cudaStream_t st);
int flow_identity_loss(const awb_prior* h, const awb_grid_spec* g, const Workspace& ws, cudaStream_t st);
// dgrid (optional, single object, use_linear): d / d grid [B,C,H,W] = linear.weight[c] * (gradient at the 1x1-conv output)
int flow_backward(const awb_prior* h, const float* params, const awb_grid_spec* g, const Workspace& ws,
                  cudaStream_t st, bool use_linear = true, float* dgrid = nullptr);
int flow_save_floats(int C);                                     // floats saved per pixel and flow by the training forward
bool flow_seg_capable(const awb_prior* h);                        // C = 2, m <= 32: segment-table kernels exist (awb_flow.cu)
bool flow_seg_path(const awb_prior* h);                           // ... and are the ones this handle runs
bool flow_seg3_capable(const awb_prior* h);                       // C = 3: forward tables for the one-masked-coordinate flows
int64_t flow_tab_floats(const awb_prior* h);                      // size of Workspace.flowtab
int64_t flow_seg_scratch_floats(const awb_prior* h, int S);       // size of Workspace.flowseg
bool flow_bwd_dz_in_smem(const awb_prior* h, int64_t N);         // the backward keeps its running gradient on the SM
int flow_actnorm_init(const awb_prior* h, float* params, const awb_grid_spec* g, const Workspace& ws,
                      cudaStream_t st);

// ---- NormalizingFlow1D coupling flow (ConvexDiffeomorphismNet), implemented in awb_diffeo.cu
int diffeo_forward(const awb_prior* h, const float* params, const awb_grid_spec* g, const Workspace& ws, float* deformed,
                   cudaStream_t st);
// dgrid (optional, single object): d / d grid [B,2,H,W] = linear.weight^T (gradient at the linear's output)
int diffeo_backward(const awb_prior* h, const float* params, const awb_grid_spec* g, const Workspace& ws, cudaStream_t st,
                    float* dgrid = nullptr);
inline bool has_flow(const awb_prior* h) { return h->desc.kind == AWB_KIND_FLOW_ICNN || h->desc.kind == AWB_KIND_DIFFEO_ICNN; }
// the coordinate transform in front of the ICNN, whichever flow the prior has
inline int any_flow_forward(const awb_prior* h, const float* params, const awb_grid_spec* g, const Workspace& ws,
                            float* deformed, cudaStream_t st) {
  return h->desc.kind == AWB_KIND_DIFFEO_ICNN ? diffeo_forward(h, params, g, ws, deformed, st)
                                              : flow_forward(h, params, g, ws, deformed, st);
}
inline int any_flow_backward(const awb_prior* h, const float* params, const awb_grid_spec* g, const Workspace& ws,
                             cudaStream_t st, float* dgrid = nullptr) {
  return h->desc.kind == AWB_KIND_DIFFEO_ICNN ? diffeo_backward(h, params, g, ws, st, dgrid)
                                              : flow_backward(h, params, g, ws, st, true, dgrid);
}

// Pixel coordinate of local row n (global row n + g.row0), channel c (SURVEY a1).  torch.linspace semantics for
// AWB_GRID_LINSPACE: step = 1/(n-1); first half start+i*step, second half end-(n-1-i)*step.
__device__ __forceinline__ float lin01(int i, int n) {
  if (n <= 1) return 0.f;
  float step = 1.0f / (float)(n - 1);
  return (i < n / 2) ? (float)i * step : 1.0f - (float)(n - 1 - i) * step;
}
__device__ __forceinline__ float coord(const GridDev& g, int64_t n, int c) {
  // 32-bit index arithmetic: N <= 2^30 pixel rows is checked at every entry point (check_common)
  const uint32_t hw = (uint32_t)g.H * (uint32_t)g.W, nn = (uint32_t)n + g.row0;
  const uint32_t b = nn / hw, r = nn - b * hw;
  if (g.mode == AWB_GRID_EXPLICIT) return g.grid[((int64_t)b * g.C + c) * hw + r];
  if (c == 2) return g.t0 + (float)b * g.t_step;
  const uint32_t i = r / (uint32_t)g.W, j = r - i * (uint32_t)g.W;
  if (g.mode == AWB_GRID_LINSPACE) return c == 0 ? lin01((int)j, g.W) : lin01((int)i, g.H);
  return c == 0 ? (float)j / (float)g.W : (float)i / (float)g.H;
}
// Index of local row n, channel c in a planar [B,C,H,W] tensor (the layout of the grid and of its gradient dgrid).
__device__ __forceinline__ int64_t planar_index(const GridDev& g, int64_t n, int c) {
  const uint32_t hw = (uint32_t)g.H * (uint32_t)g.W, nn = (uint32_t)n + g.row0;
  const uint32_t b = nn / hw, r = nn - b * hw;
  return ((int64_t)b * g.C + c) * hw + r;
}

}  // namespace awb
