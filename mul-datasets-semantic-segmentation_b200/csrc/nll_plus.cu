// nll_plus.cu — the "NLLPlus" loss path (SURVEY §8 row f4): soft-max in the UNIFIED space, bipartite projection of
// the probabilities, bilinear up-sampling (align_corners=True) of the projected probabilities, -log at the label class.
//
// Reference work replaced: AdjNLLPlusLoss.forward (lib/loss/loss_helper.py:647-668)
//     pred  = softmax(x, dim=1)                                   -> mdseg_softmax_nchw
//     probs = einsum('bchw,nc->bnhw', pred, Adj)                  -> mdseg_proj_fwd (existing)
//     probs = F.interpolate(probs, size=label HxW, bilinear, align_corners=True)
//     loss  = gather(-log(probs), label)[label != ignore]         -> mdseg_up_nll_fwd (neither [B,C,H,W] tensor exists)
// and its autograd replay, driven by MdsOhemNLLPlusLoss (lib/loss/ohem_ce_loss.py:92-146) with the same OHEM
// selection as MdsOhemCELoss.  Only the label class of a pixel enters its loss, so the per-pixel work is one
// 4-corner gather forward and one tent-weighted accumulation backward; the class-dense work is at LOW resolution.
//
// Backward: d loss / d probs_low[b, n, y, x] = sum over the label pixels p under the tent of (y, x) with label n and
// p in S of  -w * tent(p; y, x) / prob(p).  One thread per low-res corner walks its <= (2 * factor)^2 label pixels and
// adds into its own corner of the plane of each pixel's class: no atomics, fixed order, deterministic.
#include "up_ce_internal.cuh"

namespace mdseg {
namespace {

template <typename T>
__global__ void __launch_bounds__(256) softmax_nchw_kernel(const T* __restrict__ x, int C, int64_t hw, float* __restrict__ pred) {
  const int b = blockIdx.y;
  const T* xb = x + (int64_t)b * C * hw;
  float* pb = pred + (int64_t)b * C * hw;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < hw; p += (int64_t)gridDim.x * blockDim.x) {
    float m = -__int_as_float(0x7f800000);
    for (int c = 0; c < C; ++c) m = fmaxf(m, to_f32<T>(xb[(int64_t)c * hw + p]));
    float s = 0.f;
    for (int c = 0; c < C; ++c) s += __expf(to_f32<T>(xb[(int64_t)c * hw + p]) - m);
    const float inv = 1.0f / s;
    for (int c = 0; c < C; ++c) pb[(int64_t)c * hw + p] = __expf(to_f32<T>(xb[(int64_t)c * hw + p]) - m) * inv;
  }
}

// dx = pred * (dpred - sum_c pred_c dpred_c)
template <typename T>
__global__ void __launch_bounds__(256) softmax_bwd_nchw_kernel(const float* __restrict__ pred, const float* __restrict__ dpred,
                                                               int C, int64_t hw, T* __restrict__ dx) {
  const int b = blockIdx.y;
  const float* pb = pred + (int64_t)b * C * hw;
  const float* gb = dpred + (int64_t)b * C * hw;
  T* ob = dx + (int64_t)b * C * hw;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < hw; p += (int64_t)gridDim.x * blockDim.x) {
    float t = 0.f;
    for (int c = 0; c < C; ++c) t = fmaf(pb[(int64_t)c * hw + p], gb[(int64_t)c * hw + p], t);
    for (int c = 0; c < C; ++c) {
      const int64_t o = (int64_t)c * hw + p;
      ob[o] = from_f32<T>(pb[o] * (gb[o] - t));
    }
  }
}

struct NllArgs {
  mdseg_src_table src;  // projected probabilities, fp32
  mdseg_src_table dst;  // backward: d loss / d probs planes, fp32, zero-initialised by the caller
  const int32_t* dataset_ids;
  const void* labels;
  Geom gm;
  int ignore;
  float* loss_px;
  mdseg_ohem_state* states;
  const float* grad_out;
  float grad_scale;
  int* err_flag;
};

// one thread per label pixel; a CTA covers 256 consecutive pixels of one image
template <typename L>
__global__ void __launch_bounds__(256) up_nll_fwd_kernel(const NllArgs a) {
  const int b = blockIdx.y;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  const Geom& gm = a.gm;
  const int64_t ppi = (int64_t)gm.H * gm.W;
  const L* labels = (const L*)a.labels + (int64_t)b * ppi;
  float* loss = a.loss_px + (int64_t)b * ppi;
  unsigned n_valid = 0, n_hard = 0, n_px = 0;
  double sum_hard = 0.0;
  const bool valid_ds = d >= 0 && d < a.src.n_datasets;
  if (!valid_ds) {
    // image of no dataset: not part of the loss vector (sentinel -1) but its labels count in n_min (:99)
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < ppi; p += (int64_t)gridDim.x * blockDim.x) {
      loss[p] = -1.0f;
      n_valid += (load_label<L>(labels, p) != a.ignore) ? 1u : 0u;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.err_flag) atomicOr(a.err_flag, MDSEG_ERR_DATASET_ID);
    block_accumulate_stats(a.states, n_valid, 0u, 0.0, 0u);
    return;
  }
  const int C = a.src.C[d];
  const float* q = (const float*)a.src.base[d] + (int64_t)b * a.src.image_stride[d];
  mdseg_ohem_state* st = a.states + (a.src.seg_per_dataset ? d : 0);
  const float thresh = st->thresh;
  const int64_t hw = (int64_t)gm.h * gm.w;
  int err = 0;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < ppi; p += (int64_t)gridDim.x * blockDim.x) {
    const int Y = (int)(p / gm.W), X = (int)(p - (int64_t)Y * gm.W);
    const int lv = load_label<L>(labels, p);
    float l = 0.f;
    ++n_px;
    if (lv != a.ignore) {
      if ((unsigned)lv >= (unsigned)C) {
        err = 1;
      } else {
        ++n_valid;
        int y0, y1, x0, x1;
        float ly0, ly1, lx0, lx1;
        gm.ym.at(Y, y0, y1, ly0, ly1);
        gm.xm.at(X, x0, x1, lx0, lx1);
        const float* pl = q + (int64_t)lv * hw;
        const float v00 = __ldg(pl + (int64_t)y0 * gm.w + x0), v01 = __ldg(pl + (int64_t)y0 * gm.w + x1);
        const float v10 = __ldg(pl + (int64_t)y1 * gm.w + x0), v11 = __ldg(pl + (int64_t)y1 * gm.w + x1);
        // ATen's operand order (UpSampleBilinear2d): h0 * (w0 * a + w1 * b) + h1 * (w0 * c + w1 * d)
        const float pr = ly0 * (lx0 * v00 + lx1 * v01) + ly1 * (lx0 * v10 + lx1 * v11);
        l = -logf(pr);
        if (l > thresh) { ++n_hard; sum_hard += (double)l; }
      }
    }
    loss[p] = l;
  }
  if (__syncthreads_or(err) && threadIdx.x == 0 && a.err_flag) atomicOr(a.err_flag, MDSEG_ERR_LABEL_RANGE);
  block_accumulate_stats(st, n_valid, n_hard, sum_hard, n_px);
}

// one thread per low-res corner (b, y, x): gathers the label pixels under its tent
template <typename L>
__global__ void __launch_bounds__(128) up_nll_bwd_kernel(const NllArgs a) {
  const int b = blockIdx.z;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  if (d < 0 || d >= a.src.n_datasets) return;
  const Geom& gm = a.gm;
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= gm.w) return;
  const int C = a.src.C[d];
  const mdseg_ohem_state* st = a.states + (a.src.seg_per_dataset ? d : 0);
  SelParams sp;
  sp.thresh = st->thresh; sp.kth = st->kth; sp.mode = st->mode;
  sp.w = (a.grad_out ? a.grad_out[a.src.seg_per_dataset ? d : 0] : 1.f) * a.grad_scale * st->inv_n_sel;
  if (sp.w == 0.f) return;
  const int64_t ppi = (int64_t)gm.H * gm.W, hw = (int64_t)gm.h * gm.w;
  const L* labels = (const L*)a.labels + (int64_t)b * ppi;
  const float* loss = a.loss_px + (int64_t)b * ppi;
  float* dq = (float*)a.dst.base[d] + (int64_t)b * a.dst.image_stride[d] + (int64_t)y * gm.w + x;
  const int Y0 = first_dst_ge(gm.ym, y - 1, gm.H), Y1 = first_dst_ge(gm.ym, y + 1, gm.H);
  const int X0 = first_dst_ge(gm.xm, x - 1, gm.W), X1 = first_dst_ge(gm.xm, x + 1, gm.W);
  for (int Y = Y0; Y < Y1; ++Y) {
    int i0, i1;
    float l0, l1;
    gm.ym.at(Y, i0, i1, l0, l1);
    const float wy = (i0 == y ? l0 : 0.f) + (i1 == y ? l1 : 0.f);
    if (wy == 0.f) continue;
    for (int X = X0; X < X1; ++X) {
      int j0, j1;
      float m0, m1;
      gm.xm.at(X, j0, j1, m0, m1);
      const float wx = (j0 == x ? m0 : 0.f) + (j1 == x ? m1 : 0.f);
      const int64_t p = (int64_t)Y * gm.W + X;
      const int lv = load_label<L>(labels, p);
      if (wx == 0.f || lv == a.ignore || (unsigned)lv >= (unsigned)C) continue;
      const float l = loss[p];
      if (!is_selected(sp, l)) continue;
      // d(-log pr)/d pr = -1 / pr with pr = exp(-loss)
      dq[(int64_t)lv * hw] += -sp.w * wy * wx * expf(l);
    }
  }
}

template <typename L>
int launch_fwd(const NllArgs& a, int n_images, cudaStream_t s) {
  const int64_t ppi = (int64_t)a.gm.H * a.gm.W;
  int64_t bx = ceil_div64(ppi, 256);
  const int64_t want = ceil_div64((int64_t)sm_count() * 16, n_images);
  if (bx > want) bx = want;
  up_nll_fwd_kernel<L><<<dim3((unsigned)bx, (unsigned)n_images), 256, 0, s>>>(a);
  MDSEG_LAUNCH_OK();
  return 0;
}
template <typename L>
int launch_bwd(const NllArgs& a, int n_images, cudaStream_t s) {
  dim3 grid((unsigned)((a.gm.w + 127) / 128), (unsigned)a.gm.h, (unsigned)n_images);
  up_nll_bwd_kernel<L><<<grid, 128, 0, s>>>(a);
  MDSEG_LAUNCH_OK();
  return 0;
}

}  // namespace
}  // namespace mdseg

extern "C" int mdseg_softmax_nchw(const void* x, int dtype, int n_images, int C, int64_t hw, float* pred, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && C > 0 && hw >= 0, "mdseg_softmax_nchw: bad shape");
  if (n_images == 0 || hw == 0) return 0;
  MDSEG_REQUIRE(x && pred, "mdseg_softmax_nchw: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  int64_t bx = ceil_div64(hw, 256);
  if (bx > 65535) bx = 65535;
  dim3 grid((unsigned)bx, (unsigned)n_images);
  return with_float_type(dtype, "mdseg_softmax_nchw", "dtype", [&](auto t) {
    using T = typename decltype(t)::type;
    softmax_nchw_kernel<T><<<grid, 256, 0, s>>>((const T*)x, C, hw, pred);
    MDSEG_LAUNCH_OK();
    return 0;
  });
}

extern "C" int mdseg_softmax_bwd_nchw(const float* pred, const float* dpred, int n_images, int C, int64_t hw, void* dx,
                                      int dx_dtype, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && C > 0 && hw >= 0, "mdseg_softmax_bwd_nchw: bad shape");
  if (n_images == 0 || hw == 0) return 0;
  MDSEG_REQUIRE(pred && dpred && dx, "mdseg_softmax_bwd_nchw: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  int64_t bx = ceil_div64(hw, 256);
  if (bx > 65535) bx = 65535;
  dim3 grid((unsigned)bx, (unsigned)n_images);
  return with_float_type(dx_dtype, "mdseg_softmax_bwd_nchw", "dx_dtype", [&](auto t) {
    using T = typename decltype(t)::type;
    softmax_bwd_nchw_kernel<T><<<grid, 256, 0, s>>>(pred, dpred, C, hw, (T*)dx);
    MDSEG_LAUNCH_OK();
    return 0;
  });
}

extern "C" int mdseg_up_nll_fwd(const mdseg_src_table* src, const int32_t* dataset_ids, const void* labels, int label_dtype,
                                int n_images, int h, int w, int H, int W, int ignore, float* loss_px,
                                mdseg_ohem_state* states, int32_t* err_flag, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(src_count_ok(src) && src->dtype == MDSEG_F32,
                "mdseg_up_nll_fwd: the projected probabilities must be an fp32 source table");
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0 && H > 0 && W > 0, "mdseg_up_nll_fwd: bad shape");
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(labels && loss_px && states, "mdseg_up_nll_fwd: null pointer");
  NllArgs a;
  a.src = *src; a.dst = *src; a.dataset_ids = dataset_ids; a.labels = labels; a.gm = make_geom(h, w, H, W);
  a.ignore = ignore; a.loss_px = loss_px; a.states = states; a.grad_out = nullptr; a.grad_scale = 1.f;
  a.err_flag = err_flag;
  cudaStream_t s = (cudaStream_t)stream;
  return with_int_type(label_dtype, "mdseg_up_nll_fwd", "label dtype",
                       [&](auto l) { return launch_fwd<typename decltype(l)::type>(a, n_images, s); });
}

extern "C" int mdseg_up_nll_bwd(const mdseg_src_table* src, const int32_t* dataset_ids, const void* labels, int label_dtype,
                                int n_images, int h, int w, int H, int W, int ignore, const float* loss_px,
                                const mdseg_ohem_state* states, const float* grad_out, float grad_scale,
                                const mdseg_src_table* dst, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(src_count_ok(src) && dst && dst->n_datasets == src->n_datasets && dst->dtype == MDSEG_F32,
                "mdseg_up_nll_bwd: bad source / destination table");
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && h <= 65535 && w > 0 && H > 0 && W > 0,
                "mdseg_up_nll_bwd: bad shape");
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(labels && loss_px && states, "mdseg_up_nll_bwd: null pointer");
  NllArgs a;
  a.src = *src; a.dst = *dst; a.dataset_ids = dataset_ids; a.labels = labels; a.gm = make_geom(h, w, H, W);
  a.ignore = ignore; a.loss_px = const_cast<float*>(loss_px); a.states = const_cast<mdseg_ohem_state*>(states);
  a.grad_out = grad_out; a.grad_scale = grad_scale; a.err_flag = nullptr;
  cudaStream_t s = (cudaStream_t)stream;
  return with_int_type(label_dtype, "mdseg_up_nll_bwd", "label dtype",
                       [&](auto l) { return launch_bwd<typename decltype(l)::type>(a, n_images, s); });
}
