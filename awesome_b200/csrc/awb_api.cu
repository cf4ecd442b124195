// extern "C" entry points of libawb.so (declared in include/awb.h) and the host-side
// bookkeeping behind them: handle, parameter-arena layout, workspace carving, error state.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <vector>

#include "awb_internal.cuh"

namespace awb {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return AWB_ERR_CUDA;
}

static Layout make_layout(const awb_desc& d) {
  Layout L = {};
  L.C = d.C; L.h = d.h; L.L = d.L; L.F = d.F; L.m = d.m;
  L.ld = (int)round_up(d.h + d.C + 1, 8);
  L.P_icnn = (int64_t)d.h * d.C + d.h + (int64_t)d.L * ((int64_t)d.h * d.h + d.h + (int64_t)d.h * d.C) + d.h + 1 + d.C;
  L.off_icnn = 0;
  L.per_flow = 2 * ((int64_t)d.m * d.C + d.m + (int64_t)d.C * d.m + d.C) + 2 * d.C;
  L.n_lin = 0;
  if (d.kind == AWB_KIND_FLOW_ICNN) {
    // module registration order of PathConnectedNet: convex_net, flow_net, linear
    L.off_flow = L.P_icnn;
    L.P_flow = L.per_flow * d.F;
    L.off_lin = L.off_flow + L.P_flow;
    L.n_lin = 2 * d.C;
    L.P = L.off_lin + L.n_lin;
  } else if (d.kind == AWB_KIND_DIFFEO_ICNN) {
    // ConvexDiffeomorphismNet: convex_net, diffeo_net (s.0..F-1, t.0..F-1, scale.0..F-1), linear (full C x C)
    L.per_flow = 2 * (3 * (int64_t)d.m + 3) + 4;
    L.off_flow = L.P_icnn;
    L.P_flow = L.per_flow * d.F;
    L.off_lin = L.off_flow + L.P_flow;
    L.n_lin = (int64_t)d.C * d.C + d.C;
    L.P = L.off_lin + L.n_lin;
  } else if (d.kind == AWB_KIND_STAR) {   // plain state_dict-order arena, no augmented space
    L.P = (int64_t)d.h * d.h + 8 * (int64_t)d.h + 4;
    L.P_icnn = 0; L.off_flow = 0; L.P_flow = 0; L.off_lin = L.P;
  } else {
    L.off_flow = L.P_icnn; L.P_flow = 0; L.off_lin = L.P_icnn; L.P = L.P_icnn;
  }
  L.aug_in = 0;
  L.aug_layer = 4 * (int64_t)d.h;
  L.aug_out = L.aug_layer + (int64_t)d.L * d.h * L.ld;
  L.G = L.aug_out + L.ld;
  return L;
}

static int64_t align256(int64_t b) { return round_up(b, 256); }

// fit_only: on a tensor-path handle the fused kernel keeps activations on the SM, so the [N][ld] activation / delta
// planes of the CUDA-core path are not carved (0.85 GB per 640x480 frame).
// deform_only: no ICNN partials, planes or tensor-path image either.
Workspace carve(const awb_prior* h, int64_t N, int layout, void* base) {
  const bool training = layout != AWB_WS_INFERENCE, fit_only = layout == AWB_WS_FIT_STEP,
             deform_only = layout == AWB_WS_DEFORMATION, tangent = layout == AWB_WS_SECOND_ORDER;
  const Layout& L = h->lay;
  const int64_t O = h->desc.n_objects;
  int S = n_splits(N);
  if (h->desc.precision == AWB_PREC_F16) {   // the tensor path writes one partial per CTA = per 128-pixel tile, up to 148
    int64_t t = (N + 127) / 128;
    int st = (int)(t < kMaxSplits ? t : kMaxSplits);
    if (st > S) S = st;
  }
  char* p = (char*)base;
  int64_t off = 0;
  auto take = [&](int64_t bytes) { char* r = p ? p + off : nullptr; off += align256(bytes); return r; };
  Workspace w = {};
  w.row0 = 0; w.N = N;
  if (h->desc.kind == AWB_KIND_STAR) {   // AWB_WS_FIT_STEP only (check_common): the fit kernel's per-CTA partials
    const int Ss = star_bwd_ctas(N, nullptr);
    w.part = (float*)take(4 * (int64_t)Ss * L.P);
    w.lossp = (float*)take(4 * (int64_t)Ss);
    w.bytes = off;
    return w;
  }
  w.waug = (float*)take(4 * O * L.G);
  w.part = (float*)take(training && !deform_only ? 4 * (int64_t)S * O * L.G : 0);
  w.lossp = (float*)take(4 * ((int64_t)kMaxSplits * O + O));   // [S][O] loss partials + [O] spare scalars (max |dlogits|)
  w.fpart = (float*)take(training ? 4 * (int64_t)S * O * (L.P_flow + L.n_lin) : 0);
  w.X = (float*)take(4 * O * N * 4);
  w.dX = (float*)take(training ? 4 * O * N * 4 : 0);
  const bool planes = !deform_only && !(fit_only && h->desc.precision == AWB_PREC_F16 && tc_supported(h));
  w.ZA = (float*)take(planes ? 4 * O * (L.L + 1) * N * L.ld : 0);
  w.D = (float*)take(training && planes ? 4 * O * 2 * N * L.ld : 0);
  w.logits = (float*)take(4 * O * N);
  const bool rnvp = h->desc.kind == AWB_KIND_FLOW_ICNN;
  w.flowz = (float*)take(training ? 4 * O * N * (int64_t)L.F * (rnvp ? flow_save_floats(L.C) : L.C) : 0);
  if (!training || L.F == 0) w.flowz = nullptr;
  w.flowd = (training && rnvp && L.C == 3 && !flow_bwd_dz_in_smem(h, N)) ? (float*)take(4 * O * N * 4) : nullptr;
  w.flowtab = (rnvp && flow_tab_floats(h) > 0) ? (float*)take(4 * flow_tab_floats(h)) : nullptr;
  w.flowseg = (training && rnvp && flow_seg_scratch_floats(h, S) > 0) ? (float*)take(4 * flow_seg_scratch_floats(h, S)) : nullptr;
  w.tc = (!deform_only && h->desc.precision == AWB_PREC_F16 && tc_supported(h)) ? (void*)take(O * (int64_t)tc_image_bytes(L.L))
                                                                               : nullptr;
  w.ZT = tangent ? (float*)take(4 * O * (L.L + 1) * N * L.ld) : nullptr;
  w.bytes = off;
  w.row0 = 0; w.N = N;
  return w;
}

}  // namespace awb

using namespace awb;

extern "C" {

const char* awb_version(void) { return "awb 0.1 (sm_100a)"; }
const char* awb_last_error(void) { return g_err; }

int awb_prior_create(const awb_desc* d, awb_handle* out) {
  if (!d || !out) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (d->kind != AWB_KIND_ICNN && d->kind != AWB_KIND_FLOW_ICNN && d->kind != AWB_KIND_STAR && d->kind != AWB_KIND_DIFFEO_ICNN) { set_error("unknown prior kind %d", d->kind); return AWB_ERR_INVALID; }
  if (d->kind == AWB_KIND_STAR && (d->C != 2 || d->h > 160 || d->n_objects != 1 || d->precision != AWB_PREC_FP32)) {
    set_error("star prior: C = 2, n_hidden <= 160, one object, fp32");
    return AWB_ERR_UNSUPPORTED;
  }
  if (d->C < 2 || d->C > 3) { set_error("C must be 2 or 3, got %d", d->C); return AWB_ERR_UNSUPPORTED; }
  if (d->h < 8 || d->h > 256) { set_error("h must be in [8,256], got %d", d->h); return AWB_ERR_UNSUPPORTED; }
  if (d->L < 0 || d->L > 8) { set_error("L must be in [0,8], got %d", d->L); return AWB_ERR_UNSUPPORTED; }
  if (d->n_objects < 1 || d->n_objects > 16) { set_error("n_objects must be in [1,16], got %d", d->n_objects); return AWB_ERR_UNSUPPORTED; }
  if (d->kind == AWB_KIND_DIFFEO_ICNN && (d->C != 2 || d->m < 1 || d->m > 96 || (d->F != 2 && d->F != 4 && d->F != 6 && d->F != 8))) {
    set_error("NormalizingFlow1D needs C=2, num_coupling in {2,4,6,8} and width <= 96, got C=%d F=%d m=%d", d->C, d->F, d->m);
    return AWB_ERR_UNSUPPORTED;
  }
  if (d->kind == AWB_KIND_FLOW_ICNN && (d->F < 1 || d->F > 64 || d->m < 1 || d->m > 32)) {
    set_error("flow needs 1<=F<=64 and 1<=m<=32, got F=%d m=%d", d->F, d->m);
    return AWB_ERR_UNSUPPORTED;
  }
  if (d->precision != AWB_PREC_FP32 && d->precision != AWB_PREC_F16) { set_error("unknown precision %d", d->precision); return AWB_ERR_INVALID; }
  awb_prior* h = new awb_prior();
  h->desc = *d;
  if (d->kind == AWB_KIND_ICNN || d->kind == AWB_KIND_STAR) { h->desc.F = 0; h->desc.m = 0; }
  if (d->kind == AWB_KIND_STAR) h->desc.L = 0;
  h->lay = make_layout(h->desc);
  h->fc_set = false;
  h->fc.out_scale = 1.f;
  h->flow_eval = 0;
  h->d_map = nullptr; h->d_clamp = nullptr; h->d_group = nullptr; h->d_tcmap = nullptr; h->d_imap = nullptr; h->d_aug2img = nullptr;
  const Layout& L = h->lay;
  // arena (state_dict order) -> augmented index; clamp mask; optimizer groups
  std::vector<int32_t> map(L.P_icnn);
  std::vector<uint8_t> clamp(L.P, 0), group(L.P, 1);
  int64_t i = 0;
  const int hh = L.h, C = L.C, ld = L.ld;
  if (d->kind != AWB_KIND_STAR) {
  for (int j = 0; j < hh; j++) for (int c = 0; c < C; c++) map[i++] = (int32_t)(L.aug_in + j * 4 + c);  // input.weight
  for (int j = 0; j < hh; j++) map[i++] = (int32_t)(L.aug_in + j * 4 + 3);                               // input.bias
  for (int l = 0; l < L.L; l++) {
    int64_t base = L.aug_layer + (int64_t)l * hh * ld;
    for (int j = 0; j < hh; j++) for (int k = 0; k < hh; k++) { clamp[L.off_icnn + i] = 1; map[i++] = (int32_t)(base + (int64_t)j * ld + k); }  // ln.weight
    for (int j = 0; j < hh; j++) map[i++] = (int32_t)(base + (int64_t)j * ld + hh + C);                  // ln.bias
    for (int j = 0; j < hh; j++) for (int c = 0; c < C; c++) map[i++] = (int32_t)(base + (int64_t)j * ld + hh + c);  // skp.weight
  }
  for (int k = 0; k < hh; k++) { clamp[L.off_icnn + i] = 1; map[i++] = (int32_t)(L.aug_out + k); }       // out.ln.weight
  map[i++] = (int32_t)(L.aug_out + hh + C);                                                             // out.ln.bias
  for (int c = 0; c < C; c++) map[i++] = (int32_t)(L.aug_out + hh + c);                                  // out.skp.weight
  }
  if (d->kind == AWB_KIND_STAR) {
    i = 0;
    group[0] = 2; group[1] = 2;                                         // offset: its own optimizer group
    const int64_t o_W2r = 2 + 3 * (int64_t)hh + (int64_t)hh * hh + hh + hh + 1 + hh + hh;
    for (int k = 0; k < hh; k++) clamp[o_W2r + k] = 1;                  // W2_r.weight >= 0 (cell 3)
  }
  if (i != L.P_icnn) { set_error("internal: layout mismatch"); awb_prior_destroy(h); return AWB_ERR_INVALID; }
  for (int64_t k = L.off_flow; k < L.off_flow + L.P_flow; k++) group[k] = 0;
  for (int64_t k = L.off_lin; k < L.P; k++) group[k] = 2;
  if (d->kind == AWB_KIND_DIFFEO_ICNN) {
    // weight-norm gains form their own optimizer group (3): the reference decays only `*weight_g`
    // (awesome/util/torch.py:19-35, convex_diffeomorphism_net.py "weight_decay_on_weight_g")
    const int64_t bsz = 3 * (int64_t)d->m + 3;
    for (int b = 0; b < 2 * d->F; b++) {
      group[L.off_flow + b * bsz + d->m] = 3;
      group[L.off_flow + b * bsz + 2 * d->m + 2] = 3;
    }
    for (int i = 0; i < d->F; i++) group[L.off_flow + 2 * d->F * bsz + 4 * i + 2] = 3;
  }
  std::vector<int32_t> imap(L.G, -1);
  for (int64_t k = 0; k < L.P_icnn; k++) imap[map[k]] = (int32_t)k;
  cudaError_t e;
  auto fail = [&](const char* what) { awb_prior_destroy(h); return cuda_fail(e, what); };   // frees what was allocated
  if ((e = cudaMalloc(&h->d_imap, sizeof(int32_t) * L.G)) != cudaSuccess ||
      (e = cudaMemcpy(h->d_imap, imap.data(), sizeof(int32_t) * L.G, cudaMemcpyHostToDevice)) != cudaSuccess)
    return fail("awb_prior_create (inverse map)");
  if ((e = cudaGetDevice(&h->device)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_map, sizeof(int32_t) * L.P_icnn)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_clamp, L.P)) != cudaSuccess || (e = cudaMalloc(&h->d_group, L.P)) != cudaSuccess ||
      (e = cudaMemcpy(h->d_map, map.data(), sizeof(int32_t) * L.P_icnn, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(h->d_clamp, clamp.data(), L.P, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(h->d_group, group.data(), L.P, cudaMemcpyHostToDevice)) != cudaSuccess)
    return fail("awb_prior_create");
  if (d->kind != AWB_KIND_STAR && tc_supported(h)) {
    std::vector<int32_t> tmap(tc_map_elems(L.L)), a2i(L.G);
    tc_build_map_host(L, tmap.data());
    tc_build_aug2img_host(L, a2i.data());
    if ((e = cudaMalloc(&h->d_tcmap, sizeof(int32_t) * tmap.size())) != cudaSuccess ||
        (e = cudaMemcpy(h->d_tcmap, tmap.data(), sizeof(int32_t) * tmap.size(), cudaMemcpyHostToDevice)) != cudaSuccess ||
        (e = cudaMalloc(&h->d_aug2img, sizeof(int32_t) * L.G)) != cudaSuccess ||
        (e = cudaMemcpy(h->d_aug2img, a2i.data(), sizeof(int32_t) * L.G, cudaMemcpyHostToDevice)) != cudaSuccess)
      return fail("awb_prior_create (tensor path)");
  } else if (d->precision == AWB_PREC_F16) {
    awb_prior_destroy(h);
    set_error("precision f16 (tcgen05 path) supports priors with ICNN width h=130 and L in {1,2}; use fp32 for this shape");
    return AWB_ERR_UNSUPPORTED;
  }
  *out = h;
  return AWB_OK;
}

int awb_prior_destroy(awb_handle h) {
  if (!h) return AWB_OK;
  cudaFree(h->d_map); cudaFree(h->d_clamp); cudaFree(h->d_group); cudaFree(h->d_tcmap); cudaFree(h->d_imap); cudaFree(h->d_aug2img);
  if (h->stream_made) {
    cudaStreamDestroy(h->copy_stream);
    for (int b = 0; b < 2; b++) { cudaEventDestroy(h->ev_ready[b]); cudaEventDestroy(h->ev_free[b]); }
  }
  delete h;
  return AWB_OK;
}

int64_t awb_prior_param_count(awb_handle h) { return h ? h->lay.P : -1; }

int64_t awb_prior_workspace_bytes(awb_handle h, int64_t n_pixels, int32_t layout) {
  if (!h || n_pixels < 1 || layout < AWB_WS_INFERENCE || layout > AWB_WS_SECOND_ORDER) return -1;
  if (h->desc.kind == AWB_KIND_STAR && layout != AWB_WS_FIT_STEP) return -1;   // the star prior has only the fit step
  return carve(h, n_pixels, layout, nullptr).bytes;
}

int64_t awb_opt_state_bytes(awb_handle h) {
  if (!h) return -1;
  int64_t n = h->lay.P * h->desc.n_objects;
  return round_up(2 * n * 4, 256) + round_up((int64_t)sizeof(OptScal) * h->desc.n_objects, 256);
}

int awb_prior_set_flow_consts(awb_handle h, const float* nmin, const float* nmax, float new_min, float new_max,
                              const uint8_t* masks) {
  if (!h || !nmin || !nmax || !masks) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (h->desc.kind != AWB_KIND_FLOW_ICNN) { set_error("not a flow prior"); return AWB_ERR_INVALID; }
  for (int c = 0; c < h->lay.C; c++) { h->fc.nmin[c] = nmin[c]; h->fc.nmax[c] = nmax[c]; }
  h->fc.new_min = new_min; h->fc.new_max = new_max;
  memcpy(h->fc.masks, masks, (size_t)h->lay.F * h->lay.C);
  h->fc_set = true;
  return AWB_OK;
}

int awb_prior_set_flow_output_scale(awb_handle h, float scale) {
  if (!h) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (h->desc.kind != AWB_KIND_FLOW_ICNN) { set_error("not a flow prior"); return AWB_ERR_INVALID; }
  if (!(scale > 0.f) || !isfinite(scale)) { set_error("output_scale must be a positive finite number"); return AWB_ERR_INVALID; }
  h->fc.out_scale = scale;
  return AWB_OK;
}

int awb_prior_set_flow_eval(awb_handle h, int32_t mode) {
  if (!h) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (h->desc.kind != AWB_KIND_FLOW_ICNN) { set_error("not a flow prior"); return AWB_ERR_INVALID; }
  if (mode < 0 || mode > 2) { set_error("flow_eval must be 0 (auto), 1 (unit loops) or 2 (segment tables), got %d", mode); return AWB_ERR_INVALID; }
  if (mode == 2 && !flow_seg_capable(h) && !flow_seg3_capable(h)) { set_error("segment tables need m <= 32"); return AWB_ERR_UNSUPPORTED; }
  h->flow_eval = mode;
  return AWB_OK;
}

// A star handle reaches the generic entry points only through the whole-batch fit step (awb_prior_fit_step, _fit_steps,
// _fit_host_frames); every other one refuses it here, before anything reads its layout as an ICNN's.
static int refuse_star() {
  set_error("the star prior runs awb_star_forward / awb_star_backward on points and awb_prior_fit_step (or _fit_steps, "
            "_fit_host_frames) on an explicit grid; this entry point does not take star handles");
  return AWB_ERR_UNSUPPORTED;
}

// Validates the arguments every workspace entry point shares and carves the workspace, of layout `layout` (AWB_WS_*),
// into *out.  window (optional, {row_begin, row_end}): the call works on the pixel rows [row_begin, row_end) of the
// batch, which must be a non-empty range inside [0, N), and the workspace is sized for them; out->row0 = row_begin.
static int check_common(awb_handle h, const awb_grid_spec* g, void* ws, size_t ws_bytes, int layout,
                        const int64_t* window, Workspace* out) {
  if (h && h->desc.kind == AWB_KIND_STAR && (layout != AWB_WS_FIT_STEP || window)) return refuse_star();
  if (!h || !g || !ws) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (g->B < 1 || g->H < 1 || g->W < 1) { set_error("empty grid %dx%dx%d", g->B, g->H, g->W); return AWB_ERR_INVALID; }
  if (g->mode == AWB_GRID_EXPLICIT && !g->grid) { set_error("explicit grid needs a pointer"); return AWB_ERR_INVALID; }
  if (g->mode < 0 || g->mode > 2) { set_error("unknown grid mode %d", g->mode); return AWB_ERR_INVALID; }
  const int64_t N = (int64_t)g->B * g->H * g->W;
  if (N > (int64_t)1 << 30) { set_error("too many pixel rows"); return AWB_ERR_UNSUPPORTED; }
  if (window && (window[0] < 0 || window[0] >= window[1] || window[1] > N)) {
    set_error("pixel-row window [%lld, %lld) is empty or outside [0, %lld)", (long long)window[0], (long long)window[1],
              (long long)N);
    return AWB_ERR_INVALID;
  }
  const Workspace w = carve(h, window ? window[1] - window[0] : N, layout, ws);
  if ((int64_t)ws_bytes < w.bytes) { set_error("workspace too small: %lld < %lld", (long long)ws_bytes, (long long)w.bytes); return AWB_ERR_WORKSPACE; }
  if (h->desc.kind == AWB_KIND_FLOW_ICNN && !h->fc_set) { set_error("awb_prior_set_flow_consts not called"); return AWB_ERR_INVALID; }
  *out = w;
  out->row0 = window ? window[0] : 0;
  return AWB_OK;
}

static bool loss_weighted(const awb_loss_spec* loss, int O) {
  for (int o = 0; o < O; o++)
    if (loss_is_weighted(loss[o])) return true;
  return false;
}

// The per-pixel part of the loss specs of a fit step: an ignore label must be a number (NaN never equals a target).
static int check_loss(const awb_loss_spec* loss, int O) {
  for (int o = 0; o < O; o++)
    if (loss[o].ignore_enabled && !isfinite(loss[o].ignore_value)) {
      set_error("loss[%d]: ignore_value must be finite", o);
      return AWB_ERR_INVALID;
    }
  return AWB_OK;
}

// One pass of an ICNN prior on the rows of a workspace.  dy comes from the loss on target (fit step: forward and
// backward), from dlogits (backward of an earlier training forward on the same workspace, which holds the flow's outputs
// and, on the exact path, the ICNN's activations) or from nowhere (forward only).
struct Pass {
  bool tensor;                                      // the fused tcgen05 kernel, else the exact fp32 kernels
  const float* target; const awb_loss_spec* loss;   // dy from the loss on target ...
  const float* dlogits;                             // ... or dy = dlogits
  float *logits, *deformed, *dgrid;                 // optional outputs (a plain ICNN leaves dgrid in ws.dX)
  bool training;                                    // exact forward only: keep the activations for a later backward
  bool reuse;                                       // tensor path: the packed fp16 weight image in ws is current
};

// Flow forward, ICNN on the chosen path, flow backward.  The flow always runs on CUDA cores (K = C is too thin for
// tensor cores): it writes the deformed coordinates X that the ICNN reads and consumes the d / d X the ICNN returns.
// *n_part: the number of ICNN gradient partials written.
static int run_pass(awb_handle h, const float* params, const awb_grid_spec* g, const Workspace& w, const Pass& p,
                    cudaStream_t st, int* n_part) {
  const bool flow = has_flow(h), forward = !p.dlogits, backward = p.target || p.dlogits;
  const bool need_dx = backward && (flow || p.dgrid);
  int rc;
  if (flow && forward) {
    rc = any_flow_forward(h, params, g, w, p.deformed, st);   // keeps X (and the coupling inputs when training)
    if (rc) return rc;
  }
  if (p.tensor) {
    // backward from dlogits: the fused kernel recomputes the forward and reads dy as the target of an upstream "loss"
    const int O = h->desc.n_objects;
    awb_loss_spec up[16] = {};
    float* amax = nullptr;
    float* wamax = nullptr;
    if (p.dlogits) {
      for (int o = 0; o < O && o < 16; o++) { up[o].kind = AWB_LOSS_UPSTREAM; up[o].cls_rule = AWB_CLS_UNARY_LT_HALF; up[o].coef_fg = 1.f; up[o].coef_bg = 1.f; }
      amax = w.lossp + (int64_t)kMaxSplits * O;       // spare floats behind the loss partials (lossp is [S][O], S <= 148 ... see carve)
      rc = absmax_per_object(p.dlogits, w.N, O, amax, st);
      if (rc) return rc;
    } else if (p.target && loss_weighted(p.loss, O)) {
      wamax = w.lossp + (int64_t)kMaxSplits * O;      // the same spare floats: max |w| over the kept pixels
      rc = weight_absmax_per_object(p.loss, p.target, w.N, O, wamax, st);
      if (rc) return rc;
    }
    *n_part = 0;
    rc = tc_fit_forward_backward(h, params, g, p.dlogits ? p.dlogits : p.target, p.dlogits ? up : p.loss, p.logits,
                                 backward ? 1 : 0, w, n_part, st, p.reuse, flow ? w.X : nullptr,
                                 need_dx ? w.dX : nullptr, amax, wamax);
  } else {
    *n_part = n_splits(w.N);
    rc = forward ? simt_forward(h, params, g, p.logits, p.training || backward, flow, w, st) : AWB_OK;
    if (!rc && backward) rc = simt_backward(h, p.target, p.loss, p.dlogits, need_dx, w, st);
  }
  if (rc) return rc;
  // flow priors: the flow backward writes dgrid itself (dX holds the gradient at the deformed coordinates, not the grid)
  return flow && backward ? any_flow_backward(h, params, g, w, st, p.dgrid) : AWB_OK;
}

int awb_prior_forward(awb_handle h, const float* params, const awb_grid_spec* g, float* logits, float* deformed,
                      int32_t mode, void* ws, size_t ws_bytes, void* stream) {
  if (mode < AWB_FWD_EXACT || mode > AWB_FWD_TC_TRAINING) { set_error("unknown forward mode %d", mode); return AWB_ERR_INVALID; }
  const bool training = mode == AWB_FWD_EXACT_TRAINING || mode == AWB_FWD_TC_TRAINING;
  const bool tensor = mode == AWB_FWD_TC || mode == AWB_FWD_TC_TRAINING;   // the default forward stays exact fp32
  Workspace w;
  int rc = check_common(h, g, ws, ws_bytes, training ? AWB_WS_TRAINING : AWB_WS_INFERENCE, nullptr, &w);
  if (rc) return rc;
  if (!params) { set_error("null params"); return AWB_ERR_INVALID; }
  if (tensor && h->desc.precision != AWB_PREC_F16) { set_error("tensor-path forward needs an f16 handle"); return AWB_ERR_INVALID; }
  if (tensor && !logits) { set_error("null logits"); return AWB_ERR_INVALID; }
  Pass p = {};
  p.tensor = tensor; p.logits = logits; p.deformed = deformed; p.training = training;
  int n_part;
  return run_pass(h, params, g, w, p, (cudaStream_t)stream, &n_part);
}

int awb_prior_flow_inverse(awb_handle h, const float* params, const awb_grid_spec* g, float* out, void* stream) {
  if (h && h->desc.kind == AWB_KIND_STAR) return refuse_star();
  if (!h || !params || !g || !out) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (h->desc.kind != AWB_KIND_FLOW_ICNN || !h->fc_set) { set_error("needs a flow prior with its constants set"); return AWB_ERR_INVALID; }
  if (g->mode != AWB_GRID_EXPLICIT || !g->grid || g->B < 1 || g->H < 1 || g->W < 1) { set_error("inverse takes an explicit [B,C,H,W] tensor"); return AWB_ERR_INVALID; }
  return flow_inverse(h, params, g, out, (cudaStream_t)stream);
}

int awb_prior_backward(awb_handle h, const float* params, const awb_grid_spec* g, const float* dlogits, float* grads,
                       float* dgrid, void* ws, size_t ws_bytes, void* stream) {
  Workspace w;
  int rc = check_common(h, g, ws, ws_bytes, AWB_WS_TRAINING, nullptr, &w);
  if (rc) return rc;
  if (!params || !dlogits || !grads) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (dgrid && (h->desc.kind == AWB_KIND_STAR || h->desc.n_objects != 1)) {
    set_error("dgrid is provided for single-object ICNN, RealNVP o ICNN and NormalizingFlow1D o ICNN priors only "
              "(no caller needs it on grouped or star handles; kind %d, %d objects)", h->desc.kind, h->desc.n_objects);
    return AWB_ERR_UNSUPPORTED;
  }
  cudaStream_t st = (cudaStream_t)stream;
  // the path follows the handle, not the forward: an f16 handle's backward is the fused tensor-path kernel even after an
  // exact training forward
  Pass p = {};
  p.tensor = h->desc.precision == AWB_PREC_F16; p.dlogits = dlogits; p.dgrid = dgrid;
  int n_part;
  rc = run_pass(h, params, g, w, p, st, &n_part);
  if (rc) return rc;
  rc = simt_reduce_grads(h, grads, w, w.N, st, n_part);
  if (rc) return rc;
  return dgrid && !has_flow(h) ? simt_dgrid(h, g, dgrid, w, st) : AWB_OK;   // plain ICNN: dX is d / d grid
}

int awb_prior_grid_grad_backward(awb_handle h, const float* params, const awb_grid_spec* g, const float* dlogits,
                                 const float* d_dgrid, float* d_dlogits, float* grads, void* ws, size_t ws_bytes,
                                 void* stream) {
  if (!h) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (h->desc.kind == AWB_KIND_STAR) return refuse_star();
  if (h->desc.kind != AWB_KIND_ICNN || h->desc.n_objects != 1) {
    set_error("the second-order pass is provided for single-object ICNN priors only (kind %d, %d objects)", h->desc.kind,
              h->desc.n_objects);
    return AWB_ERR_UNSUPPORTED;
  }
  Workspace w;
  int rc = check_common(h, g, ws, ws_bytes, AWB_WS_SECOND_ORDER, nullptr, &w);
  if (rc) return rc;
  if (!params || !dlogits || !d_dgrid || !d_dlogits || !grads) { set_error("null argument"); return AWB_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  rc = simt_grid_grad_backward(h, g, dlogits, d_dgrid, d_dlogits, w, st);
  if (rc) return rc;
  return simt_reduce_grads(h, grads, w, w.N, st, n_splits(w.N));
}

int awb_prior_fit_step(awb_handle h, float* params, void* opt_state, const awb_grid_spec* g, const float* target,
                       const awb_loss_spec* loss, const awb_opt_hyper* hy, float* loss_out, void* ws, size_t ws_bytes,
                       int32_t flags, void* stream) {
  Workspace w;
  int rc = check_common(h, g, ws, ws_bytes, AWB_WS_FIT_STEP, nullptr, &w);
  if (rc) return rc;
  if (!params || !opt_state || !target || !loss || !hy) { set_error("null argument"); return AWB_ERR_INVALID; }
  if ((rc = check_loss(loss, h->desc.n_objects))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (h->desc.kind == AWB_KIND_STAR) {   // k_star_bwd<NU, WL> over the grid's rows; no packed image, so flags do not apply
    if (g->mode != AWB_GRID_EXPLICIT) { set_error("a star fit step takes an explicit [B,2,H,W] grid"); return AWB_ERR_INVALID; }
    int S = 0;
    rc = star_fit(h, params, g, target, *loss, w, &S, st);
    if (rc) return rc;
    return reduce_opt_plain(h, params, opt_state, hy, loss_out, w.part, S, h->lay.P, w.lossp, 1, st);
  }
  // simt_reduce_opt refreshes a flow prior's fp16 weight image only when its optimizer owns every group
  Pass p = {};
  p.tensor = h->desc.precision == AWB_PREC_F16; p.target = target; p.loss = loss;
  p.reuse = (flags & AWB_FIT_REUSE_PACKED) != 0 && (!has_flow(h) || hy->active_groups == 0);
  int n_part;
  rc = run_pass(h, params, g, w, p, st, &n_part);
  if (rc) return rc;
  return simt_reduce_opt(h, params, opt_state, hy, loss_out, w, w.N, st, n_part);
}

// get_deformation: single-object RealNVP o ICNN and NormalizingFlow1D o ICNN handles
static int check_deformable(awb_handle h) {
  if (!h) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (h->desc.kind == AWB_KIND_STAR) return refuse_star();
  if (h->desc.kind == AWB_KIND_ICNN) { set_error("an ICNN prior has no deformation"); return AWB_ERR_INVALID; }
  if (!has_flow(h) || h->desc.n_objects != 1) {
    set_error("the deformation entry points support single-object flow priors (kind %d, %d objects)", h->desc.kind,
              h->desc.n_objects);
    return AWB_ERR_UNSUPPORTED;
  }
  return AWB_OK;
}

int awb_prior_deformation(awb_handle h, const float* params, const awb_grid_spec* g, float* deformed, int32_t training,
                          void* ws, size_t ws_bytes, void* stream) {
  int rc = check_deformable(h);
  if (rc) return rc;
  Workspace w;
  rc = check_common(h, g, ws, ws_bytes, AWB_WS_DEFORMATION, nullptr, &w);
  if (rc) return rc;
  if (!params || !deformed) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (!training) w.flowz = nullptr;   // the coupling records are kept for awb_prior_deformation_backward only
  return any_flow_forward(h, params, g, w, deformed, (cudaStream_t)stream);
}

int awb_prior_deformation_backward(awb_handle h, const float* params, const awb_grid_spec* g, const float* d_deformed,
                                   float* grads, float* dgrid, void* ws, size_t ws_bytes, void* stream) {
  int rc = check_deformable(h);
  if (rc) return rc;
  Workspace w;
  rc = check_common(h, g, ws, ws_bytes, AWB_WS_DEFORMATION, nullptr, &w);
  if (rc) return rc;
  if (!params || !d_deformed || !grads) { set_error("null argument"); return AWB_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  rc = simt_seed_dX(h, d_deformed, w, st);
  if (rc) return rc;
  rc = any_flow_backward(h, params, g, w, st, dgrid);
  if (rc) return rc;
  return simt_reduce_grads(h, grads, w, w.N, st, /*n_partials=*/0);   // no ICNN partials: its entries are exactly 0
}

// PathConnectedNet.inverse with autograd: single-object RealNVP o ICNN handles, explicit grid; carves layout
// AWB_WS_DEFORMATION
static int check_inverse(awb_handle h, const awb_grid_spec* g, void* ws, size_t ws_bytes, Workspace* w) {
  if (h && h->desc.kind == AWB_KIND_STAR) return refuse_star();
  if (!h || !g) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (h->desc.kind != AWB_KIND_FLOW_ICNN) { set_error("needs a flow prior with its constants set"); return AWB_ERR_INVALID; }
  if (h->desc.n_objects != 1) {
    set_error("the inverse entry points support single-object flow priors (%d objects)", h->desc.n_objects);
    return AWB_ERR_UNSUPPORTED;
  }
  if (g->mode != AWB_GRID_EXPLICIT) { set_error("inverse takes an explicit [B,C,H,W] tensor"); return AWB_ERR_INVALID; }
  return check_common(h, g, ws, ws_bytes, AWB_WS_DEFORMATION, nullptr, w);
}

int awb_prior_inverse(awb_handle h, const float* params, const awb_grid_spec* g, float* out, int32_t training,
                      void* ws, size_t ws_bytes, void* stream) {
  Workspace w;
  int rc = check_inverse(h, g, ws, ws_bytes, &w);
  if (rc) return rc;
  if (!params || !out) { set_error("null argument"); return AWB_ERR_INVALID; }
  return flow_inverse(h, params, g, out, (cudaStream_t)stream, training ? &w : nullptr);
}

int awb_prior_inverse_backward(awb_handle h, const float* params, const awb_grid_spec* g, const float* d_out,
                               float* grads, float* dgrid, void* ws, size_t ws_bytes, void* stream) {
  Workspace w;
  int rc = check_inverse(h, g, ws, ws_bytes, &w);
  if (rc) return rc;
  if (!params || !d_out || !grads) { set_error("null argument"); return AWB_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  rc = flow_inverse_backward(h, params, g, w, d_out, dgrid, st);
  if (rc) return rc;
  return simt_reduce_grads(h, grads, w, w.N, st, /*n_partials=*/0);   // no ICNN partials: its entries are exactly 0
}

// single-object ICNN and RealNVP o ICNN handles (the priors of the spatio-temporal fit)
static int check_sliceable(awb_handle h) {
  if (!h) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (h->desc.kind == AWB_KIND_STAR) return refuse_star();
  if ((h->desc.kind != AWB_KIND_ICNN && h->desc.kind != AWB_KIND_FLOW_ICNN) || h->desc.n_objects != 1) {
    set_error("gradient rows support single-object ICNN and RealNVP o ICNN priors (kind %d, %d objects)", h->desc.kind,
              h->desc.n_objects);
    return AWB_ERR_UNSUPPORTED;
  }
  return AWB_OK;
}

int64_t awb_prior_grad_row_floats(awb_handle h) { return h ? h->lay.P + 1 : -1; }

int awb_prior_slice_grads(awb_handle h, const float* params, const awb_grid_spec* g, int64_t row_begin, int64_t row_end,
                          const float* target, const awb_loss_spec* loss, float* grad_row, void* ws, size_t ws_bytes,
                          int32_t flags, void* stream) {
  int rc = check_sliceable(h);
  if (rc) return rc;
  Workspace w;
  const int64_t window[2] = {row_begin, row_end};
  rc = check_common(h, g, ws, ws_bytes, AWB_WS_FIT_STEP, window, &w);
  if (rc) return rc;
  if (!params || !target || !loss || !grad_row) { set_error("null argument"); return AWB_ERR_INVALID; }
  if ((rc = check_loss(loss, 1))) return rc;
  awb_loss_spec ls = *loss;              // the weight map, like the target, is the full batch's: read at the global row
  if (ls.weight) ls.weight += row_begin;
  Pass p = {};
  p.tensor = h->desc.precision == AWB_PREC_F16; p.target = target + row_begin; p.loss = &ls;
  p.reuse = (flags & AWB_FIT_REUSE_PACKED) != 0;
  cudaStream_t st = (cudaStream_t)stream;
  int n_part;
  rc = run_pass(h, params, g, w, p, st, &n_part);
  if (rc) return rc;
  return simt_reduce_grads(h, grad_row, w, w.N, st, n_part, grad_row + h->lay.P);   // the loss sum goes to column P
}

int awb_prior_rows_opt_step(awb_handle h, float* params, void* opt_state, const float* rows, int32_t n_rows,
                            const awb_opt_hyper* hy, float* loss_out, void* ws, size_t ws_bytes, void* stream) {
  (void)ws; (void)ws_bytes;   // the optimizer needs no scratch (see awb.h)
  int rc = check_sliceable(h);
  if (rc) return rc;
  if (!params || !opt_state || !rows || !hy) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (n_rows < 1) { set_error("n_rows must be >= 1, got %d", n_rows); return AWB_ERR_INVALID; }
  const int64_t R = h->lay.P + 1;
  return reduce_opt_plain(h, params, opt_state, hy, loss_out, rows, n_rows, R, rows + h->lay.P, R, (cudaStream_t)stream);
}

int awb_prior_fit_steps(awb_handle h, float* params, void* opt_state, const awb_grid_spec* g, const float* const* targets,
                        int32_t n_targets, int32_t first, int32_t n_steps, const awb_loss_spec* loss, const awb_opt_hyper* hy,
                        float* loss_out, void* ws, size_t ws_bytes, int32_t flags, void* stream) {
  if (!targets || n_targets < 1 || n_steps < 0 || first < 0) { set_error("bad target list"); return AWB_ERR_INVALID; }
  for (int i = 0; i < n_targets; i++)
    if (!targets[i]) { set_error("targets[%d] is null", i); return AWB_ERR_INVALID; }
  const int O = h ? h->desc.n_objects : 1;
  for (int s = 0; s < n_steps; s++) {
    int rc = awb_prior_fit_step(h, params, opt_state, g, targets[(first + s) % n_targets], loss, hy,
                                loss_out ? loss_out + (size_t)s * O : nullptr, ws, ws_bytes,
                                (s > 0 || (flags & AWB_FIT_REUSE_PACKED)) ? AWB_FIT_REUSE_PACKED : 0, stream);
    if (rc) return rc;
  }
  return AWB_OK;
}

int awb_prior_fit_host_frames(awb_handle h, float* params, void* opt_state, const awb_grid_spec* g,
                              const float* const* host_targets, int32_t n_host, int32_t n_steps, const awb_loss_spec* loss,
                              const awb_opt_hyper* hy, float* loss_host, float* staging, void* ws, size_t ws_bytes,
                              int32_t flags, void* stream) {
  Workspace w;   // awb_prior_fit_step carves it again for every step
  int rc = check_common(h, g, ws, ws_bytes, AWB_WS_FIT_STEP, nullptr, &w);
  if (rc) return rc;
  const int64_t N = w.N;
  if (!params || !opt_state || !host_targets || !loss || !hy || !staging) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (n_host < 1 || n_steps < 0) { set_error("n_host must be >= 1 and n_steps >= 0"); return AWB_ERR_INVALID; }
  for (int i = 0; i < n_host; i++)
    if (!host_targets[i]) { set_error("host_targets[%d] is null", i); return AWB_ERR_INVALID; }
  float* loss_dev = nullptr;
  if (loss_host) {   // the optimizer kernel stores each step's loss straight into mapped host memory
    cudaPointerAttributes at;
    AWB_CUDA(cudaPointerGetAttributes(&at, loss_host));
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) {
      set_error("loss_host must be pinned (cudaHostAlloc / cudaHostRegister) host memory");
      return AWB_ERR_INVALID;
    }
    loss_dev = (float*)at.devicePointer;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (!h->stream_made) {
    AWB_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    for (int b = 0; b < 2; b++) {
      AWB_CUDA(cudaEventCreateWithFlags(&h->ev_ready[b], cudaEventDisableTiming));
      AWB_CUDA(cudaEventCreateWithFlags(&h->ev_free[b], cudaEventDisableTiming));
    }
    h->stream_made = true;
  }
  const int O = h->desc.n_objects;
  const size_t frame_bytes = (size_t)O * N * sizeof(float);
  // the staging buffers may still be read by work queued on `st` before this call
  AWB_CUDA(cudaEventRecord(h->ev_free[0], st));
  AWB_CUDA(cudaStreamWaitEvent(h->copy_stream, h->ev_free[0], 0));
  for (int s = 0; s < n_steps; s++) {
    const int b = s & 1;
    float* dst = staging + (size_t)b * O * N;
    if (s >= 2) AWB_CUDA(cudaStreamWaitEvent(h->copy_stream, h->ev_free[b], 0));   // step s-2 has consumed this buffer
    AWB_CUDA(cudaMemcpyAsync(dst, host_targets[s % n_host], frame_bytes, cudaMemcpyHostToDevice, h->copy_stream));
    AWB_CUDA(cudaEventRecord(h->ev_ready[b], h->copy_stream));
    AWB_CUDA(cudaStreamWaitEvent(st, h->ev_ready[b], 0));
    rc = awb_prior_fit_step(h, params, opt_state, g, dst, loss, hy, loss_dev ? loss_dev + (size_t)s * O : nullptr, ws, ws_bytes,
                            (s > 0 || (flags & AWB_FIT_REUSE_PACKED)) ? AWB_FIT_REUSE_PACKED : 0, stream);
    if (rc) return rc;
    AWB_CUDA(cudaEventRecord(h->ev_free[b], st));
  }
  return AWB_OK;
}

int awb_flow_identity_step(awb_handle h, float* params, void* opt_state, const awb_grid_spec* g,
                           const awb_opt_hyper* hy, float* loss_out, void* ws, size_t ws_bytes, void* stream) {
  Workspace w;
  int rc = check_common(h, g, ws, ws_bytes, AWB_WS_TRAINING, nullptr, &w);
  if (rc) return rc;
  if (!params || !opt_state || !hy) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (h->desc.kind != AWB_KIND_FLOW_ICNN) { set_error("not a flow prior"); return AWB_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  rc = flow_forward(h, params, g, w, nullptr, st, /*use_linear=*/false);
  if (rc) return rc;
  rc = flow_identity_loss(h, g, w, st);
  if (rc) return rc;
  rc = flow_backward(h, params, g, w, st, /*use_linear=*/false);
  if (rc) return rc;
  awb_opt_hyper hh = *hy;
  hh.active_groups = 1;   // flow_net only
  return simt_reduce_opt(h, params, opt_state, &hh, loss_out, w, w.N, st, n_splits(w.N));
}

int awb_optim_step(awb_handle h, float* params, const float* grads, void* opt_state, const awb_opt_hyper* hy,
                   void* stream) {
  if (!h || !params || !grads || !opt_state || !hy) { set_error("null argument"); return AWB_ERR_INVALID; }
  return optim_step(h, params, grads, opt_state, hy, (cudaStream_t)stream);
}

int awb_prior_enforce_convexity(awb_handle h, float* params, void* stream) {
  if (!h || !params) { set_error("null argument"); return AWB_ERR_INVALID; }
  return clamp_only(h, params, (cudaStream_t)stream);
}

int awb_opt_state_init(awb_handle h, void* opt_state, const double* lr, void* stream) {
  if (!h || !opt_state || !lr) { set_error("null argument"); return AWB_ERR_INVALID; }
  return opt_state_init(h, opt_state, lr, (cudaStream_t)stream);
}

int awb_star_forward(awb_handle h, const float* params, const float* x, int64_t n, float* logits, void* stream) {
  if (!h || !params || !x || !logits || n < 1) { set_error("bad argument"); return AWB_ERR_INVALID; }
  if (h->desc.kind != AWB_KIND_STAR) { set_error("not a star prior"); return AWB_ERR_INVALID; }
  return star_run(h, params, x, nullptr, n, nullptr, logits, nullptr, nullptr, false, nullptr, (cudaStream_t)stream);
}

int64_t awb_star_workspace_bytes(awb_handle h, int64_t n) {
  if (!h || n < 1 || h->desc.kind != AWB_KIND_STAR) return -1;
  const int S = star_n_ctas(n);
  return round_up(4 * (int64_t)S * h->lay.P, 256) + round_up(4 * (int64_t)S, 256);
}

int awb_star_fit_step(awb_handle h, float* params, void* opt_state, const float* x, const float* target, int64_t n,
                      const awb_loss_spec* loss, const awb_opt_hyper* hy, float* loss_out, void* ws, size_t ws_bytes,
                      void* stream) {
  if (!h || !params || !opt_state || !x || !target || !loss || !hy || !ws || n < 1) { set_error("bad argument"); return AWB_ERR_INVALID; }
  if (h->desc.kind != AWB_KIND_STAR) { set_error("not a star prior"); return AWB_ERR_INVALID; }
  if (loss_is_weighted(*loss)) {
    set_error("awb_star_fit_step takes no weight map or ignore label; awb_prior_fit_step with an explicit [1,2,1,n] grid "
              "of the sampled points takes both");
    return AWB_ERR_UNSUPPORTED;
  }
  const int64_t need = awb_star_workspace_bytes(h, n);
  if ((int64_t)ws_bytes < need) { set_error("workspace too small: %lld < %lld", (long long)ws_bytes, (long long)need); return AWB_ERR_WORKSPACE; }
  const int S = star_n_ctas(n);
  float* part = (float*)ws;
  float* lossp = (float*)((char*)ws + round_up(4 * (int64_t)S * h->lay.P, 256));
  int nc = 0;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = star_run(h, params, x, target, n, loss, nullptr, part, lossp, true, &nc, st);
  if (rc) return rc;
  return reduce_opt_plain(h, params, opt_state, hy, loss_out, part, nc, h->lay.P, lossp, 1, st);
}

int64_t awb_star_backward_workspace_bytes(awb_handle h, int64_t n) {
  if (!h || n < 1 || h->desc.kind != AWB_KIND_STAR) return -1;
  return round_up(4 * (int64_t)star_bwd_ctas(n, nullptr) * h->lay.P, 256);
}

int awb_star_backward(awb_handle h, const float* params, const float* x, int64_t n, const float* dlogits, float* grads,
                      float* dx, void* ws, size_t ws_bytes, void* stream) {
  if (!h || !params || !x || !dlogits || !grads || !ws || n < 1) { set_error("bad argument"); return AWB_ERR_INVALID; }
  if (h->desc.kind != AWB_KIND_STAR) { set_error("not a star prior"); return AWB_ERR_INVALID; }
  const int64_t need = awb_star_backward_workspace_bytes(h, n);
  if ((int64_t)ws_bytes < need) { set_error("workspace too small: %lld < %lld", (long long)ws_bytes, (long long)need); return AWB_ERR_WORKSPACE; }
  return star_backward(h, params, x, dlogits, n, grads, dx, (float*)ws, (cudaStream_t)stream);
}

int awb_opt_set_lr(awb_handle h, void* opt_state, const double* lr, void* stream) {
  if (!h || !opt_state || !lr) { set_error("null argument"); return AWB_ERR_INVALID; }
  return opt_set_lr(h, opt_state, lr, (cudaStream_t)stream);
}

int awb_opt_plateau_step(awb_handle h, void* opt_state, const float* loss, int32_t loss_stride, const awb_opt_hyper* hy,
                         void* stream) {
  if (!h || !opt_state || !loss || !hy) { set_error("null argument"); return AWB_ERR_INVALID; }
  if (loss_stride != 0 && loss_stride != 1) { set_error("loss_stride must be 0 (shared scalar) or 1 ([O])"); return AWB_ERR_INVALID; }
  return plateau_step(h, opt_state, loss, loss_stride, hy, (cudaStream_t)stream);
}

int awb_opt_read_scalars(awb_handle h, const void* opt_state, int32_t obj, awb_opt_scalars* out, void* stream) {
  if (!h || !opt_state || !out || obj < 0 || obj >= h->desc.n_objects) { set_error("bad argument"); return AWB_ERR_INVALID; }
  int64_t n = h->lay.P * h->desc.n_objects;
  const OptScal* sc = (const OptScal*)((const char*)opt_state + round_up(2 * n * 4, 256)) + obj;
  OptScal s;
  AWB_CUDA(cudaMemcpyAsync(&s, sc, sizeof(s), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  AWB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  out->step = s.step; out->num_bad = s.num_bad; out->nonfinite = s.nonfinite; out->pad = 0;
  for (int g = 0; g < AWB_MAX_GROUPS; g++) out->lr[g] = s.lr[g];
  out->best = s.best; out->last_loss = s.last_loss; out->pad2 = 0.f;
  return AWB_OK;
}

int awb_prior_actnorm_init(awb_handle h, float* params, const awb_grid_spec* g, void* ws, size_t ws_bytes,
                           void* stream) {
  Workspace w;
  int rc = check_common(h, g, ws, ws_bytes, AWB_WS_INFERENCE, nullptr, &w);
  if (rc) return rc;
  if (h->desc.kind != AWB_KIND_FLOW_ICNN) { set_error("not a flow prior"); return AWB_ERR_INVALID; }
  return flow_actnorm_init(h, params, g, w, (cudaStream_t)stream);
}

}  // extern "C"
