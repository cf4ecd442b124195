// Per-kernel-class timing with CUDA events on the launching stream, and a launch counter.
// Used by bench.py for the roofline (average duration of the dominant kernel, measured live) and for
// its gpu_launches claim.  Timing is off by default; the counter is always on.
#include <stdlib.h>

#include "awb_internal.cuh"

namespace awb {

static const int kMaxRec = 256;
static const char* kNames[PK_COUNT] = {"pack", "input_layer", "gemm_fwd", "out_loss", "gemm_wgrad", "gemm_dgrad",
                                       "input_bwd", "reduce_opt", "flow_fwd", "flow_bwd", "tc_fused", "misc",
                                       "tangent_fwd", "tangent_out"};
static struct Prof {
  bool on = false;
  cudaEvent_t ev[PK_COUNT][kMaxRec][2];
  int n[PK_COUNT] = {0};
  bool made = false;
  long long launches = 0;
  long long per_class[PK_COUNT] = {0};
} g;

// Programmatic dependent launch of the fit-step kernels is on unless AWB_NO_PDL is set (A/B measurements).
bool pdl_enabled() {
  static const bool on = getenv("AWB_NO_PDL") == nullptr;
  return on;
}

void prof_begin(int cls, cudaStream_t st) {
  g.launches++;
  g.per_class[cls]++;
  if (!g.on || g.n[cls] >= kMaxRec) return;
  cudaEventRecord(g.ev[cls][g.n[cls]][0], st);
}

void prof_end(int cls, cudaStream_t st) {
  if (!g.on || g.n[cls] >= kMaxRec) return;
  cudaEventRecord(g.ev[cls][g.n[cls]][1], st);
  g.n[cls]++;
}

}  // namespace awb

using namespace awb;

extern "C" {

int awb_profile_enable(int32_t on) {
  if (on && !g.made) {
    for (int c = 0; c < PK_COUNT; c++)
      for (int i = 0; i < kMaxRec; i++)
        for (int k = 0; k < 2; k++) AWB_CUDA(cudaEventCreate(&g.ev[c][i][k]));
    g.made = true;
  }
  for (int c = 0; c < PK_COUNT; c++) g.n[c] = 0;
  g.on = on != 0;
  return AWB_OK;
}

int awb_profile_classes(void) { return PK_COUNT; }
const char* awb_profile_class_name(int32_t cls) { return (cls >= 0 && cls < PK_COUNT) ? kNames[cls] : ""; }

int awb_profile_read(double* total_ms, int32_t* counts) {
  if (!total_ms || !counts) { set_error("null argument"); return AWB_ERR_INVALID; }
  AWB_CUDA(cudaDeviceSynchronize());
  for (int c = 0; c < PK_COUNT; c++) {
    double t = 0.0;
    for (int i = 0; i < g.n[c]; i++) {
      float ms = 0.f;
      AWB_CUDA(cudaEventElapsedTime(&ms, g.ev[c][i][0], g.ev[c][i][1]));
      t += ms;
    }
    total_ms[c] = t;
    counts[c] = g.n[c];
  }
  return AWB_OK;
}

long long awb_launch_count(void) { return g.launches; }

}  // extern "C"
