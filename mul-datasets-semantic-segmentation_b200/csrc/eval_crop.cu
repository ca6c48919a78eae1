// eval_crop.cu — the sliding-window evaluator MscEvalCrop (evaluate.py:650-753): probability accumulation of a chip into
// the padded scale-level map, and the bilinear resize + accumulation of a scale-level map into the label-size map.
//
// Reference work replaced per chip (evaluate.py:684-690, :706-710):
//     prob = net(crop)[0].softmax(dim=1)
//     if flip: prob += net(flip(crop))[0].flip(dims=(3,)).softmax(dim=1);  prob = torch.exp(prob)      (sic, :689)
//     prob_map[:, :, stH:endH, stW:endW] += prob
// and per scale (:722-724):  probs += F.interpolate(prob_map[window], (H, W), mode='bilinear', align_corners=True)
// The arg-max + confusion matrix that follow are mdseg_argmax_hist.
#include "common.cuh"

namespace mdseg {
namespace {

// one thread per chip pixel; classes walked three times (max, sum, write) from L1 / L2
template <typename T>
__global__ void __launch_bounds__(256) chip_accum_kernel(const T* __restrict__ lg, const T* __restrict__ lg_flip, int C,
                                                        int ch, int cw, float* __restrict__ probs, int PH, int PW, int y0,
                                                        int x0, int exp_after) {
  const int64_t n = (int64_t)ch * cw;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
    const int y = (int)(p / cw), x = (int)(p - (int64_t)y * cw);
    const int64_t pf = (int64_t)y * cw + (cw - 1 - x);  // the flipped pass is mirrored back
    float m = -__int_as_float(0x7f800000), mf = m;
    for (int c = 0; c < C; ++c) {
      m = fmaxf(m, to_f32<T>(lg[(int64_t)c * n + p]));
      if (lg_flip) mf = fmaxf(mf, to_f32<T>(lg_flip[(int64_t)c * n + pf]));
    }
    float s = 0.f, sf = 0.f;
    for (int c = 0; c < C; ++c) {
      s += __expf(to_f32<T>(lg[(int64_t)c * n + p]) - m);
      if (lg_flip) sf += __expf(to_f32<T>(lg_flip[(int64_t)c * n + pf]) - mf);
    }
    const float inv = 1.f / s, invf = lg_flip ? 1.f / sf : 0.f;
    float* dst = probs + (int64_t)(y0 + y) * PW + (x0 + x);
    for (int c = 0; c < C; ++c) {
      float v = __expf(to_f32<T>(lg[(int64_t)c * n + p]) - m) * inv;
      if (lg_flip) v += __expf(to_f32<T>(lg_flip[(int64_t)c * n + pf]) - mf) * invf;
      if (exp_after) v = expf(v);
      dst[(int64_t)c * PH * PW] += v;
    }
  }
}

// dst[c, Y, X] (+)= bilinear(align_corners=True) of the window [y0, y0 + sh) x [x0, x0 + sw) of src[c] ([PH, PW])
__global__ void __launch_bounds__(256) prob_resize_accum_kernel(const float* __restrict__ src, int C, int PH, int PW, int y0,
                                                               int x0, int sh, int sw, float* __restrict__ dst, int H, int W,
                                                               int first, float ys, float xs) {
  AxisMap ym, xm;
  ym.scale = ys; ym.n_in = sh;
  xm.scale = xs; xm.n_in = sw;
  const int64_t n = (int64_t)H * W;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
    const int Y = (int)(p / W), X = (int)(p - (int64_t)Y * W);
    int i0, i1, j0, j1;
    float l0, l1, m0, m1;
    ym.at(Y, i0, i1, l0, l1);
    xm.at(X, j0, j1, m0, m1);
    const int64_t o00 = (int64_t)(y0 + i0) * PW + x0 + j0, o01 = (int64_t)(y0 + i0) * PW + x0 + j1;
    const int64_t o10 = (int64_t)(y0 + i1) * PW + x0 + j0, o11 = (int64_t)(y0 + i1) * PW + x0 + j1;
    for (int c = 0; c < C; ++c) {
      const float* s = src + (int64_t)c * PH * PW;
      const float v = l0 * (m0 * s[o00] + m1 * s[o01]) + l1 * (m0 * s[o10] + m1 * s[o11]);
      float* d = dst + (int64_t)c * n + p;
      *d = first ? v : *d + v;
    }
  }
}

}  // namespace
}  // namespace mdseg

extern "C" int mdseg_eval_chip_accum(const void* logits, const void* logits_flip, int dtype, int C, int ch, int cw,
                                     float* probs, int PH, int PW, int y0, int x0, int exp_after, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(C > 0 && ch > 0 && cw > 0 && PH > 0 && PW > 0 && y0 >= 0 && x0 >= 0 && y0 + ch <= PH && x0 + cw <= PW,
                "mdseg_eval_chip_accum: the chip must lie inside the probability map");
  MDSEG_REQUIRE(logits && probs, "mdseg_eval_chip_accum: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  int64_t bx = ceil_div64((int64_t)ch * cw, 256);
  if (bx > 8 * (int64_t)sm_count()) bx = 8 * (int64_t)sm_count();
  return with_float_type(dtype, "mdseg_eval_chip_accum", "dtype", [&](auto t) {
    using T = typename decltype(t)::type;
    chip_accum_kernel<T><<<(unsigned)bx, 256, 0, s>>>((const T*)logits, (const T*)logits_flip, C, ch, cw, probs, PH, PW,
                                                      y0, x0, exp_after);
    MDSEG_LAUNCH_OK();
    return 0;
  });
}

extern "C" int mdseg_prob_resize_accum(const float* src, int C, int PH, int PW, int y0, int x0, int sh, int sw, float* dst,
                                       int H, int W, int first, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(C > 0 && sh > 0 && sw > 0 && y0 >= 0 && x0 >= 0 && y0 + sh <= PH && x0 + sw <= PW && H > 0 && W > 0,
                "mdseg_prob_resize_accum: the window must lie inside the source map");
  MDSEG_REQUIRE(src && dst, "mdseg_prob_resize_accum: null pointer");
  int64_t bx = ceil_div64((int64_t)H * W, 256);
  if (bx > 8 * (int64_t)sm_count()) bx = 8 * (int64_t)sm_count();
  prob_resize_accum_kernel<<<(unsigned)bx, 256, 0, (cudaStream_t)stream>>>(src, C, PH, PW, y0, x0, sh, sw, dst, H, W, first,
                                                                           axis_scale(sh, H), axis_scale(sw, W));
  MDSEG_LAUNCH_OK();
  return 0;
}
