// up_ce_internal.cuh — types shared by the generic (up_ce.cu) and the TMA-pipelined
// (up_ce_tma.cu) fused upsample + cross-entropy kernels.
#pragma once

#include "common.cuh"

namespace mdseg {

struct Geom {
  AxisMap ym, xm;
  int h, w, H, W;
};

inline Geom make_geom(int h, int w, int H, int W) {
  Geom g;
  g.ym.scale = axis_scale(h, H); g.ym.n_in = h;
  g.xm.scale = axis_scale(w, W); g.xm.n_in = w;
  g.h = h; g.w = w; g.H = H; g.W = W;
  return g;
}

// smallest dst in [0, n_out] whose source floor is >= target (n_out if none)
__device__ __forceinline__ int first_dst_ge(const AxisMap& m, int target, int n_out) {
  if (target <= 0) return 0;
  if (target > m.n_in - 1 || m.scale <= 0.f) return n_out;
  int d = (int)ceilf((float)target / m.scale);
  d = d < 0 ? 0 : (d > n_out ? n_out : d);
  while (d > 0 && m.floor_at(d - 1) >= target) --d;
  while (d < n_out && m.floor_at(d) < target) ++d;
  return d;
}

struct SelParams {
  float thresh, kth, w;
  unsigned mode;
};
// Membership in S is a pure function of the stored loss: in top-k mode
// mdseg_ohem_select has already demoted the ties that did not make the quota
// to just below kth, so `loss >= kth` is exact.
__device__ __forceinline__ bool is_selected(const SelParams& p, float loss) {
  return p.mode == 0 ? (loss > p.thresh) : (loss >= p.kth);
}

struct FwdArgs {
  mdseg_src_table src;
  const int32_t* dataset_ids;
  const void* labels;
  Geom gm;
  int ignore;
  int cc_max;  // classes per staged chunk (generic kernel)
  int fwp;     // smem row pitch (generic kernel)
  float* loss_px;
  float* lse_px;
  mdseg_ohem_state* states;
  int* err_flag;
};

struct BwdArgs {
  mdseg_src_table src;
  mdseg_src_table dstA, dstB;
  const int32_t* dataset_ids;
  const void* labels;
  Geom gm;
  int ignore;
  int cc_max;
  int fwp;
  const float* loss_px;
  const float* lse_px;
  mdseg_ohem_state* states;
  const float* grad_out;
  float grad_scale;
};

// TMA-pipelined fast path (up_ce_tma.cu).  Return 0 = launched, -1 = not applicable
// (caller falls back to the generic kernel), > 0 = error (set_error called).
int up_ce_fwd_warp(const FwdArgs& a, int label_dtype, int n_images, cudaStream_t s);  // up_ce_warp.cu (uint8 labels)
int up_ce_fwd_tma(const FwdArgs& a, int label_dtype, int n_images, cudaStream_t s);
int up_ce_bwd_tma(const BwdArgs& a, int label_dtype, int n_images, cudaStream_t s);

}  // namespace mdseg
