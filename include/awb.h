/*
 * awb.h -- C-ABI of the B200-native shape-prior fitting library (libawb.so).
 *
 * Drop-in boundary for AWESOME's prior-fit hot path (SURVEY.md section 8b).  The
 * reference is pure Python/PyTorch and has no FFI of its own; each entry point
 * below states the reference interface it replaces (paths relative to the
 * reference checkout).  The Python host side (awesome_b200/) binds these with
 * ctypes and mirrors the reference's module / optimizer / loss API on top.
 *
 * Conventions
 *  - every function returns an int status: 0 ok, <0 error; awb_last_error()
 *    returns a thread-local message.  No exceptions, no abort().
 *  - all pointers named d_* / params / grads / target / workspace are DEVICE pointers to
 *    fp32 unless stated; the library borrows them for the duration of the call
 *    and never frees or retains them (torch's caching allocator stays the owner).
 *  - all work is enqueued on the given cudaStream_t (passed as void*) and is
 *    asynchronous; calls are capturable into CUDA graphs.
 *  - a non-finite loss never traps a kernel: it skips the parameter update of
 *    that step and raises a sticky device flag (awb_opt_read_scalars).
 *  - pixel rows are ordered (b, h, w) row-major, exactly like the reference's
 *    pixelize() (awesome/util/pixelize.py:30-32).
 */
#ifndef AWB_H_
#define AWB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AWB_OK 0
#define AWB_ERR_INVALID (-1)
#define AWB_ERR_UNSUPPORTED (-2)
#define AWB_ERR_CUDA (-3)
#define AWB_ERR_WORKSPACE (-4)

/* prior kinds */
#define AWB_KIND_ICNN 0      /* ConvexNextNet / ConvexNet: awesome/model/convex_net.py:177-220 */
#define AWB_KIND_FLOW_ICNN 1 /* PathConnectedNet(RealNVP o ConvexNextNet): awesome/model/path_connected_net.py:53-85 */
#define AWB_KIND_DIFFEO_ICNN 3 /* ConvexDiffeomorphismNet(Linear -> NormalizingFlow1D -> ConvexNextNet): awesome/model/convex_diffeomorphism_net.py:130-178; desc.F = num_coupling (2/4/6/8), desc.m = backbone width (<= 96), C = 2 */
#define AWB_KIND_STAR 2      /* star-shape prior myNet(h): notebooks/icml_teaser_code/star_shaped/star.ipynb cell 2 */

/* arithmetic of the hidden-layer contractions */
#define AWB_PREC_FP32 0 /* CUDA-core fp32, bit-level comparable with the reference */
#define AWB_PREC_F16 1  /* tcgen05 kind::f16 operands, fp32 accumulation in TMEM */

/* coordinate grid conventions (SURVEY 8a row a1) */
#define AWB_GRID_EXPLICIT 0 /* caller-provided [B,C,H,W] fp32 */
#define AWB_GRID_LINSPACE 1 /* x=linspace(0,1,W)[j], y=linspace(0,1,H)[i]: awesome/dataset/transformator.py:50-60 */
#define AWB_GRID_INDEX 2    /* x=j/W, y=i/H: notebooks/how_to/convexity.ipynb cell 7 */

/* per-pixel loss kinds (SURVEY 8a row a10) */
#define AWB_LOSS_SE_SIGMOID 0 /* (t - sigmoid(y))^2: awesome/measures/se.py:21-23 on WrapperModule.process_prior_output */
#define AWB_LOSS_BCE_LOGITS 1 /* BCEWithLogitsLoss: notebooks/how_to/path-connectedness.ipynb cell 9 */
#define AWB_LOSS_UPSTREAM 2   /* internal: `target` carries d loss / d logits from autograd (awb_prior_backward on the tensor path) */
#define AWB_CLS_UNARY_LT_HALF 0 /* fg = target < 0.5: awesome/measures/unaries_weighted_loss.py:35-69 */
#define AWB_CLS_NOT_ONE 1       /* fg = target != 1: how-to notebooks, cell 9 */

#define AWB_OPT_ADAM 0
#define AWB_OPT_ADAMAX 1
#define AWB_MAX_GROUPS 4

typedef struct awb_prior* awb_handle;

typedef struct awb_desc {
  int32_t kind;      /* AWB_KIND_* */
  int32_t C;         /* coordinate channels: 2 (x,y) or 3 (x,y,t) */
  int32_t h;         /* ICNN hidden width (n_hidden, default 130) */
  int32_t L;         /* number of SkipBlocks (n_hidden_layers) */
  int32_t F;         /* number of RealNVP flows (0 for AWB_KIND_ICNN) */
  int32_t m;         /* flow MLP hidden width */
  int32_t flow_tanh; /* 1: output_fn == "tanh" */
  int32_t n_objects; /* O independent priors fitted in one grouped launch (multi-object, SURVEY a13) */
  int32_t precision; /* AWB_PREC_* */
} awb_desc;

typedef struct awb_grid_spec {
  int32_t mode;      /* AWB_GRID_* */
  int32_t B, H, W;   /* frames, height, width; N = B*H*W pixel rows */
  float t0, t_step;  /* C==3 and generated grid: t of frame b = t0 + b*t_step */
  const float* grid; /* AWB_GRID_EXPLICIT: device [B,C,H,W] */
} awb_grid_spec;

/* loss = sum_n coef(t_n) * l(y_n, t_n); coef = fg(t_n) ? coef_fg : coef_bg.  The caller folds
 * any 1/N, class weights (ratio / sssdms / equal) or fg/bg means into the two coefficients. */
typedef struct awb_loss_spec {
  int32_t kind;     /* AWB_LOSS_* */
  int32_t cls_rule; /* AWB_CLS_* */
  float coef_fg, coef_bg;
} awb_loss_spec;

typedef struct awb_opt_hyper {
  int32_t kind; /* AWB_OPT_*: torch.optim.Adam / Adamax single-tensor arithmetic */
  float beta1, beta2, eps;
  float weight_decay[AWB_MAX_GROUPS]; /* per parameter group: 0 flow_net, 1 convex_net, 2 linear */
  /* ReduceLROnPlateau(mode=min, rel threshold) stepped on the loss every iteration
   * (awesome/model/path_connected_net.py:932-933,953); disabled when plateau_enabled == 0 */
  int32_t plateau_enabled;
  int32_t patience;
  float factor, threshold, min_lr, plateau_eps;
  int32_t active_groups; /* bitmask of groups this optimizer owns; 0 = all (learn_flow_identity owns only flow_net) */
} awb_opt_hyper;

/* host-readable copy of the per-object optimizer scalars */
typedef struct awb_opt_scalars {
  int32_t step;      /* optimizer steps taken */
  int32_t num_bad;   /* plateau counter */
  int32_t nonfinite; /* sticky: a step saw a NaN/Inf loss (update skipped) */
  int32_t pad;
  double lr[AWB_MAX_GROUPS];
  double best;
  float last_loss;
  float pad2;
} awb_opt_scalars;

const char* awb_version(void);
const char* awb_last_error(void);

/* Replaces the constructor prior_model_type(**prior_model_args)
 * (awesome/run/awesome_runner.py:222-236; ConvexNextNet.__init__ convex_net.py:178-201;
 * net_factory.real_nvp_path_connected_net net_factory.py:124-176). */
int awb_prior_create(const awb_desc* desc, awb_handle* out);
int awb_prior_destroy(awb_handle h);

/* workspace layouts (awb_prior_workspace_bytes) */
#define AWB_WS_INFERENCE 0    /* awb_prior_forward(AWB_FWD_EXACT or AWB_FWD_TC), awb_prior_actnorm_init */
#define AWB_WS_TRAINING 1     /* a training forward + awb_prior_backward; large enough for every awb_prior_* entry
                                 point except awb_prior_grid_grad_backward */
#define AWB_WS_FIT_STEP 2     /* awb_prior_fit_step / _fit_steps / _fit_host_frames / _slice_grads only: much smaller on
                                 tensor-path handles, whose fused kernel keeps the activations on the SM */
#define AWB_WS_DEFORMATION 3  /* awb_prior_deformation / _deformation_backward only: the flow's buffers (deformed
                                 coordinates, coupling records, their gradient and the flow's partials), no ICNN
                                 activations; about 80 MB instead of 0.85 GB for a 640x480 C = 2 frame */
#define AWB_WS_SECOND_ORDER 4 /* awb_prior_forward(AWB_FWD_EXACT_TRAINING) followed by awb_prior_backward and
                                 awb_prior_grid_grad_backward: AWB_WS_TRAINING (a prefix of this layout) plus L + 1
                                 tangent activation planes */

/* forward modes (awb_prior_forward) */
#define AWB_FWD_EXACT 0          /* exact fp32 inference; workspace AWB_WS_INFERENCE */
#define AWB_FWD_EXACT_TRAINING 1 /* exact fp32, keeps its activations for awb_prior_backward; AWB_WS_TRAINING */
#define AWB_FWD_TC 2             /* tensor-path logits only (f16 handles); AWB_WS_INFERENCE */
#define AWB_FWD_TC_TRAINING 3    /* tensor-path training forward (f16 handles); AWB_WS_TRAINING */

/* Number of trainable fp32 parameters per object, in state_dict order (SURVEY 8b). */
int64_t awb_prior_param_count(awb_handle h);
/* Bytes of scratch the caller must provide for n_pixels rows (all objects) in workspace layout `layout` (AWB_WS_*);
 * -1 for a null handle, n_pixels < 1 or an unknown layout. */
int64_t awb_prior_workspace_bytes(awb_handle h, int64_t n_pixels, int32_t layout);
/* Layout of the optimizer state: fp32 m[O][P], then fp32 v[O][P] (Adamax: the exp_inf u), then the per-object scalars at
 * byte offset round_up(8 * O * P, 256), read through awb_opt_read_scalars. */
int64_t awb_opt_state_bytes(awb_handle h);

/* MinMax buffers of NormNet (awesome/transforms/min_max.py:28-32, net_factory.py:159-165)
 * and the coupling masks [F*C] (net_factory.py:86-99); flow priors only. */
int awb_prior_set_flow_consts(awb_handle h, const float* norm_min, const float* norm_max,
                              float new_min, float new_max, const uint8_t* masks);

/* output_scale of the coupling MLPs (normflows nets.MLP(..., output_fn, output_scale), net_factory.py:104-105): s, t =
 * scale * tanh(.).  Only applied with an output_fn (flow_tanh == 1), like normflows; default 1. */
int awb_prior_set_flow_output_scale(awb_handle h, float scale);

/* How the coupling MLPs s, t = MLP([C, m, C]) of a RealNVP prior are evaluated (net_factory.py:101-113):
 *   1  unit loops: sum_k W2[k] relu(W1[k] z + b1[k]) in the reference's order of operations;
 *   2  segment tables (m <= 32; C = 2: forward and backward, C = 3: forward of the flows that mask one coordinate): with two coordinates every coupling feeds ONE scalar into its MLPs, which
 *      are then piecewise linear with m breakpoints; the breakpoints of both nets are sorted and merged once per forward and
 *      each pixel costs one 7-step search and one FMA per net (backward: 4 histogram updates instead of 4 m masked sums).  Same function, the
 *      sums reassociated: outputs agree with mode 1 to ~1e-6, a hidden unit that is active nowhere still gets an exactly
 *      zero gradient;
 *   0  (default) mode 2 on tensor-path (AWB_PREC_F16) handles that support it, mode 1 otherwise -- the fp32 path stays
 *      the arithmetic-order parity anchor.
 * Set before the first forward of a fit; forward and backward of one step must use the same mode. */
int awb_prior_set_flow_eval(awb_handle h, int32_t mode);

/* forward(grid) -> raw logits [O][N]  (ConvexNextNet.forward convex_net.py:205-214;
 * PathConnectedNet.forward path_connected_net.py:79-85).  mode: AWB_FWD_*, each with the workspace layout named at
 * its definition; an unknown mode is AWB_ERR_INVALID.  The training modes leave what awb_prior_backward needs in the
 * workspace.  deformed (optional, [O][N][C]) receives get_deformation() (path_connected_net.py:125-129).
 * The tensor-path modes need an f16 handle.  Their logits are computed
 * with fp16 operands (fp32 accumulation): |logit - exact| <= 3e-2 * max(1, |exact|) per pixel and <= 1e-3 normwise on the
 * weights of a finished 4000-step 640x480 fit (measured 2.2e-2 / 7.0e-4, 69 of 307200 mask pixels differ:
 * tests/test_gpu_full_schedule.py); masks / reported logits use AWB_FWD_EXACT.
 * AWB_FWD_TC_TRAINING: logits from the tcgen05
 * kernel, nothing kept but the flow's deformed coordinates -- awb_prior_backward then re-runs the fused
 * forward+backward kernel with the upstream gradient (joint UNet + prior step, torch_agent.py:470-492). */
int awb_prior_forward(awb_handle h, const float* params, const awb_grid_spec* grid, float* logits,
                      float* deformed, int32_t mode, void* workspace, size_t workspace_bytes,
                      void* stream);

/* PathConnectedNet.inverse (path_connected_net.py:86-122): maps get_deformation() outputs back to grid coordinates
 * (inverse flow, inverse MinMax, inverse 1x1 conv).  grid: the deformed coordinates as [B,C,H,W]
 * (AWB_GRID_EXPLICIT); out: device [O][N][C] pixel rows. */
int awb_prior_flow_inverse(awb_handle h, const float* params, const awb_grid_spec* grid, float* out, void* stream);

/* autograd backward of forward(): dlogits [O][N] -> grads [O][P] (overwritten), optional
 * dgrid [B,C,H,W] = d loss / d grid (model_input_requires_grad configs, gradient penalties).  Must follow
 * awb_prior_forward(AWB_FWD_EXACT_TRAINING, or AWB_FWD_TC_TRAINING on f16 handles) on the same workspace.
 * dgrid is provided for single-object AWB_KIND_ICNN, AWB_KIND_FLOW_ICNN (C = 2, 3) and AWB_KIND_DIFFEO_ICNN handles, at
 * both precisions and under every flow_eval mode; the flow backward forms it in its last pass over each pixel range
 * (linear^T times the gradient at the 1x1 conv / linear output), so requesting it leaves grads bit-identical.  Grouped
 * handles (n_objects > 1) and star handles: AWB_ERR_UNSUPPORTED. */
int awb_prior_backward(awb_handle h, const float* params, const awb_grid_spec* grid,
                       const float* dlogits, float* grads, float* dgrid, void* workspace,
                       size_t workspace_bytes, void* stream);

/* Double backward of awb_prior_backward's dgrid (gradient penalties trained through the prior, DESIGN 3b.1).  The first
 * backward maps (w = dlogits, params) to dgrid_n = w_n J_n^T with J_n = d y_n / d x_n.  For the cotangent
 * d_dgrid = d R / d dgrid ([B,C,H,W], the layout of dgrid) this returns d_dlogits [N] = J_n u_n, the derivative of each
 * logit along its u_n, and grads [P] (overwritten, state_dict order) = sum_n w_n d(J_n u_n) / d params; every bias
 * entry is exactly 0.  d R / d grid is 0: the ICNN is piecewise linear in its input.  Exact fp32 kernels at both
 * precisions; the masks, weights and activations are those of the training forward.
 * Must follow awb_prior_forward(AWB_FWD_EXACT_TRAINING) on the same workspace, of layout AWB_WS_SECOND_ORDER (the
 * AWB_WS_TRAINING layout followed by L + 1 tangent activation planes).  The forward's activations are only read, so the
 * call may be repeated; awb_prior_backward may run on the same workspace before or after it.  dlogits: the first
 * backward's [N]; params: those of the forward.  Single-object AWB_KIND_ICNN handles; any other handle:
 * AWB_ERR_UNSUPPORTED. */
int awb_prior_grid_grad_backward(awb_handle h, const float* params, const awb_grid_spec* grid, const float* dlogits,
                                 const float* d_dgrid, float* d_dlogits, float* grads, void* workspace,
                                 size_t workspace_bytes, void* stream);

/* get_deformation() alone (path_connected_net.py:125-129, convex_diffeomorphism_net.py:180-185): the 1x1 conv (linear)
 * and the flow, no ICNN.  deformed: device [N][C] pixel rows.  training != 0 keeps the coupling records in the workspace
 * for awb_prior_deformation_backward.  workspace: layout AWB_WS_DEFORMATION.
 * Single-object AWB_KIND_FLOW_ICNN and AWB_KIND_DIFFEO_ICNN handles; an ICNN handle has no deformation (AWB_ERR_INVALID),
 * any other handle: AWB_ERR_UNSUPPORTED. */
int awb_prior_deformation(awb_handle h, const float* params, const awb_grid_spec* grid, float* deformed, int32_t training,
                          void* workspace, size_t workspace_bytes, void* stream);
/* Backward of awb_prior_deformation: d_deformed [N][C] (upstream gradient on the deformed coordinates) -> grads [P]
 * (overwritten, state_dict order: the flow and linear entries, every ICNN entry exactly 0) and optional dgrid [B,C,H,W].
 * Must follow awb_prior_deformation(training != 0) on the same workspace and params.  Same handles and errors. */
int awb_prior_deformation_backward(awb_handle h, const float* params, const awb_grid_spec* grid, const float* d_deformed,
                                   float* grads, float* dgrid, void* workspace, size_t workspace_bytes, void* stream);

/* One fused fit step = the body of the reference's hot loops
 * (path_connected_net.py:939-953, :364-379; notebooks/how_to/convexity.ipynb cell 9):
 * forward, sigmoid/loss, backward, cross-pixel gradient reduction, Adam/Adamax (+L2),
 * enforce_convexity clamp (convex_net.py:151-154,216-220), ReduceLROnPlateau.step(loss).
 * target [O][N]; loss/lr per object; loss_out (optional) device [O].
 * flags: AWB_FIT_REUSE_PACKED -- the previous call on this workspace was a fit step of the same handle on the same
 * params and nothing has written params since (the caller is inside its own step loop): the tensor path then
 * reuses the fp16 weight image its optimizer kernel left in the workspace instead of re-packing it. */
#define AWB_FIT_REUSE_PACKED 1
int awb_prior_fit_step(awb_handle h, float* params, void* opt_state, const awb_grid_spec* grid,
                       const float* target, const awb_loss_spec* loss, const awb_opt_hyper* hyper,
                       float* loss_out, void* workspace, size_t workspace_bytes, int32_t flags, void* stream);

/* Pixel-sliced fit step (one prior fitted on several GPUs, each computing some pixel slices of every step).
 * Single-object AWB_KIND_ICNN and AWB_KIND_FLOW_ICNN handles, both precisions; other handles: AWB_ERR_UNSUPPORTED.
 * A gradient row holds the gradient of a slice in state_dict order followed by the slice's loss sum: P + 1 floats. */
int64_t awb_prior_grad_row_floats(awb_handle h);
/* Gradient row of pixel rows [row_begin, row_end) of the batch described by grid (the reference's step restricted to
 * those pixels): forward, loss, backward, cross-CTA reduction; NO optimizer.  Coordinates (generated or read from an
 * explicit grid) are those of the global rows.  target: the FULL batch [N] (read at row_begin); loss: coefficients of the
 * FULL batch (1/N, class weights), so that rows add up to the step's gradient and loss.  workspace:
 * layout AWB_WS_FIT_STEP for row_end - row_begin pixels.  flags: AWB_FIT_REUSE_PACKED -- the previous call on this
 * workspace was a slice of the same params with the same number of rows (tensor path: its fp16 weight image, whose place
 * in the workspace depends on the row count, is reused).  An empty or out-of-range
 * window: AWB_ERR_INVALID. */
int awb_prior_slice_grads(awb_handle h, const float* params, const awb_grid_spec* grid, int64_t row_begin,
                          int64_t row_end, const float* target, const awb_loss_spec* loss, float* grad_row,
                          void* workspace, size_t workspace_bytes, int32_t flags, void* stream);
/* Sum of n_rows gradient rows (row stride awb_prior_grad_row_floats), in a fixed order, then the optimizer step of
 * awb_prior_fit_step (L2, clamp, non-finite skip + sticky flag, plateau per hyper); loss_out (optional, device) = summed
 * loss.  The same rows give the same bits on every device.  workspace: unused (may be null), kept so that the optimizer
 * can later refresh the tensor path's fp16 weight image in place without an ABI change; the next
 * awb_prior_slice_grads must therefore re-pack (flags = 0). */
int awb_prior_rows_opt_step(awb_handle h, float* params, void* opt_state, const float* rows, int32_t n_rows,
                            const awb_opt_hyper* hyper, float* loss_out, void* workspace, size_t workspace_bytes,
                            void* stream);

/* n_steps fused fit steps in one call, step s fitting the DEVICE target targets[(first + s) % n_targets] ([O][N] each): the
 * reference's step loop (path_connected_net.py:939-953) without a host round trip per step.  loss_out (optional, device):
 * [n_steps][O].  Asynchronous. */
int awb_prior_fit_steps(awb_handle h, float* params, void* opt_state, const awb_grid_spec* grid,
                        const float* const* targets, int32_t n_targets, int32_t first, int32_t n_steps,
                        const awb_loss_spec* loss, const awb_opt_hyper* hyper, float* loss_out, void* workspace,
                        size_t workspace_bytes, int32_t flags, void* stream);

/* The same loop with HOST inputs: n_steps fused fit steps, step s fitting the host frame host_targets[s % n_host]
 * ([O][N] fp32 unaries; the reference moves the frame's inputs to the device and evaluates them per frame,
 * path_connected_net.py:812-840, before the loop of :939-953; pretrain_unaries does `(1 - unaries).to(device)`, :439).  The host->device copy of frame s+1 runs on a copy stream
 * owned by the handle into the other half of `staging` (device, 2*O*N floats) while step s computes; every step's
 * loss [O] is stored by the optimizer kernel at loss_host + s*O (optional; pinned, device-mapped host memory), so
 * the host never blocks inside the loop.  Asynchronous: synchronise `stream` before reading loss_host. */
int awb_prior_fit_host_frames(awb_handle h, float* params, void* opt_state, const awb_grid_spec* grid,
                              const float* const* host_targets, int32_t n_host, int32_t n_steps,
                              const awb_loss_spec* loss, const awb_opt_hyper* hyper, float* loss_host,
                              float* staging, void* workspace, size_t workspace_bytes, int32_t flags, void* stream);

/* One step of PathConnectedNet.learn_flow_identity (path_connected_net.py:155-250): the NormNet-wrapped
 * flow alone (no 1x1 conv) is regressed onto its own input grid with SE("mean"); only the flow_net
 * group is updated (hyper->active_groups is forced to the flow group). */
int awb_flow_identity_step(awb_handle h, float* params, void* opt_state, const awb_grid_spec* grid,
                           const awb_opt_hyper* hyper, float* loss_out, void* workspace,
                           size_t workspace_bytes, void* stream);

/* torch.optim.Adam/Adamax(...).step() + enforce_convexity on caller-provided grads [O][P]
 * (agent loop: awesome/agent/torch_agent.py:489-492 + awesome_runner.py:294-297). */
int awb_optim_step(awb_handle h, float* params, const float* grads, void* opt_state,
                   const awb_opt_hyper* hyper, void* stream);
/* enforce_convexity() alone (convex_net.py:216-220). */
int awb_prior_enforce_convexity(awb_handle h, float* params, void* stream);

/* Optimizer / plateau state (fresh optimizer per frame: path_connected_net.py:923-933). */
int awb_opt_state_init(awb_handle h, void* opt_state, const double* lr_per_group, void* stream);
/* Overwrite the learning rates only (torch lr schedulers mutate param_group["lr"] between steps:
 * awesome/agent/torch_agent.py:308-325); moments, step counter and plateau state are kept. */
int awb_opt_set_lr(awb_handle h, void* opt_state, const double* lr_per_group, void* stream);
/* lr_scheduler.step(loss) alone: ReduceLROnPlateau on a caller-provided loss (device pointer, [O] or one scalar shared by
 * all objects when loss_stride == 0), without an optimizer step.  The spatio-temporal pretrain loop steps its scheduler
 * once per EPOCH on the epoch-mean loss (awesome/model/path_connected_net.py:719), not once per batch: its batch steps run
 * with hyper->plateau_enabled == 0 and the epoch end calls this. */
int awb_opt_plateau_step(awb_handle h, void* opt_state, const float* loss, int32_t loss_stride, const awb_opt_hyper* hyper,
                         void* stream);
/* synchronises the stream and copies the scalars of object obj to the host. */
int awb_opt_read_scalars(awb_handle h, const void* opt_state, int32_t obj, awb_opt_scalars* out,
                         void* stream);

/* ActNorm data-dependent init (normflows ActNorm.forward, first call): sets s,t of every
 * ActNorm from the pixel statistics of this grid, flow by flow. */
int awb_prior_actnorm_init(awb_handle h, float* params, const awb_grid_spec* grid, void* workspace,
                           size_t workspace_bytes, void* stream);

/* Star-shape prior (AWB_KIND_STAR; desc.h = n_hidden <= 160, desc.C = 2).  Parameters in state_dict order of the
 * notebook class: offset[1,2], W0.{weight[h,2],bias}, W1.{weight[h,h],bias}, W2.{weight[1,h],bias},
 * W1_r.{weight[h,1],bias}, W2_r.{weight[1,h],bias}.  x: device [n][2] sample points, logits: device [n]. */
int awb_star_forward(awb_handle h, const float* params, const float* x, int64_t n, float* logits, void* stream);
int64_t awb_star_workspace_bytes(awb_handle h, int64_t n);
/* One step of the notebook's training loop (cell 3): y = net(x); loss = sum_n coef(t_n) * l(y_n, t_n) (MSE on the
 * sigmoid with coef = 1/n in the notebook); backward; Adam/Adamax; W2_r.weight <- relu(W2_r.weight).  Optimizer
 * groups: 1 = network weights, 2 = offset (frozen until hyper->active_groups includes bit 2, cell 3 "epoch == 1000"). */
int awb_star_fit_step(awb_handle h, float* params, void* opt_state, const float* x, const float* target, int64_t n,
                      const awb_loss_spec* loss, const awb_opt_hyper* hyper, float* loss_out, void* workspace,
                      size_t workspace_bytes, void* stream);

/* counts[O][4] (int64 device): {fg&fg, pred_fg, target_fg, n} for masks thresholded at 0.5 with
 * fg = value < 0.5 (MIOU(average="binary", invert=True): awesome/measures/miou.py:29-48;
 * in-loop check path_connected_net.py:964-982). pred_is_logit: threshold logits at 0. */
int awb_mask_iou_counts(const float* pred, const float* target, int64_t n_pixels, int32_t n_objects,
                        int32_t pred_is_logit, long long* counts, void* stream);
/* target statistics for the weighted losses: counts[O][2] = {fg, bg} under cls_rule. */
int awb_target_counts(const float* target, int64_t n_pixels, int32_t n_objects, int32_t cls_rule,
                      long long* counts, void* stream);

/* Test hook: one CTA computes D[128][N] = A * B with tcgen05.mma (kind::f16, fp32 accumulate in TMEM) from raw
 * shared-memory tile images and caller-supplied descriptor fields {start offset, LBO, SBO, start advance per
 * K=16 step} (bytes).  Pins the operand-layout conventions of the tensor path against a plain matmul. */
int awb_debug_umma_probe(const void* a_bytes, int32_t a_size, const void* b_bytes, int32_t b_size, float* D,
                         int32_t N, int32_t K, int32_t a_mn_major, int32_t b_mn_major, const uint32_t* a_desc4,
                         const uint32_t* b_desc4, void* stream);

/* Debug hook: with AWB_TC_TRACE=1 in the environment the fused tensor-path kernel records clock64() stamps of its
 * pipeline stages (256 per CTA: [0,128) first epilogue thread, [128,256) MMA issuer); copies up to max_ctas CTAs of the
 * last launch to host and returns the number of CTAs copied. */
int awb_debug_tc_trace_read(unsigned long long* host, int32_t max_ctas);

/* Measurement hooks (bench.py): CUDA-event timing per kernel class on the launch stream, and the number
 * of kernels this library has launched.  awb_profile_read synchronises the device and returns, for each
 * of awb_profile_classes() classes, the summed duration [ms] and the number of timed launches. */
int awb_profile_enable(int32_t on);
int awb_profile_classes(void);
const char* awb_profile_class_name(int32_t cls);
int awb_profile_read(double* total_ms, int32_t* counts);
long long awb_launch_count(void);

/* Per-frame image preprocessing of the dataset layer on the device (SURVEY 8f N4), bit-identical to the OpenCV calls
 * the reference makes on the host.  image [n_frames][3][H][W] fp32 RGB in [0,1] (device), frames contiguous.
 * awb_image_process  = ImageSample._process_image  (awesome/dataset/image_sample.py:212-221): uint8 GaussianBlur 5x5 when
 *                      do_blur, channels reversed when bgr; out [n_frames][3][H][W], must not alias image.
 * awb_image_edge_map = ImageSample.create_edge_map (image_sample.py:260-275): out [n_frames][H][W]. */
int awb_image_process(const float* image, float* out, int32_t n_frames, int32_t H, int32_t W, int32_t do_blur, int32_t bgr,
                      void* stream);
int awb_image_edge_map(const float* image, float* out, int32_t n_frames, int32_t H, int32_t W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AWB_H_ */
