// image_pipeline.cu — the image branch of the training data pipeline in one pass (SURVEY §8 row f3).
//
// Reference work replaced, per sample, on a DataLoader worker (CPU, numpy / cv2), after im = cv2.imread(p)[:, :, ::-1]:
//   im = cv2.resize(im, (im_w, im_h))                                  RandomResizedCrop, INTER_LINEAR on uint8
//   im = np.pad(im, ((ph, ph), (pw, pw), (0, 0)))                      zero padding
//   im = im[sh:sh+crop_h, sw:sw+crop_w]; im = im[:, ::-1]              crop, RandomHorizontalFlip
//   im = contrast_table[brightness_table[im]]; im = saturate(im)       ColorJitter (brightness, contrast, saturation)
//   torch.from_numpy(im.transpose(2, 0, 1).astype(np.float32)).div_(255).sub_(mean).div_(std)     ToTensor
// as one gather: out[b, c, y, x] = norm[c][ sat_c( lut[ bilinear(src_b, Y, X) ] ) ] with the crop / pad / flip index
// map of label_pipeline.cu and colour (0, 0, 0) outside the resized image — padded pixels go through the jitter too.
// Brightness, contrast and ToTensor are functions of one byte, so the host builds them with the reference's own
// expressions (`lut`, `norm`) and the kernel only looks them up; what is computed here follows these rules exactly:
//   * INTER_LINEAR (OpenCV's fixed-point path for uint8): scale = 1 / ((double)dst / src);
//     f = (float)((d + 0.5) * scale - 0.5), s = floor(f), f -= s; weights rint((1 - f) * 2048), rint(f * 2048).
//     Columns: f = 0 and s clamped where s < 0 or s >= W - 1.  Rows: f is NOT zeroed, only both row indices are
//     clamped to [0, H - 1].  h = S[sx0] * a0 + S[sx1] * a1, out = ((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16)
//     + 2) >> 2 (VResizeLinear<uchar>).
//   * saturation: v_c = fmaf(x2, M[2][c], fmaf(x1, M[1][c], x0 * M[0][c])) / 3.0f, clipped to [0, 255], truncated —
//     the order numpy's matmul takes on x86-64.
// nvcc contracts a * b + c into an FMA unless told otherwise, so every rounding step is an explicit intrinsic.
//
// HBM-bound byte-to-float kernel: a thread produces 16 consecutive output pixels of a row, reads go through L1
// (neighbouring outputs share source bytes).  Algorithmic bytes per output pixel: 12 + (source bytes touched).
#include "common.cuh"

namespace mdseg {
namespace {

constexpr int kPx = 16;  // output pixels per thread
static_assert(sizeof(mdseg_image_view) == 328, "mdseg_image_view layout changed: update native.ImageView");

// OpenCV's INTER_LINEAR taps of output index d on an axis of `src` source samples.
struct Taps {
  int s0, s1, w0, w1;
};
__device__ __forceinline__ Taps linear_taps(int d, double scale, int src, bool zero_border) {
  float f = __double2float_rn(__dsub_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), 0.5));
  int s = (int)floorf(f);
  f = __fsub_rn(f, (float)s);
  Taps t;
  if (zero_border) {
    if (s < 0) f = 0.f, s = 0;
    if (s >= src - 1) f = 0.f, s = src - 1;
  }
  t.s0 = min(max(s, 0), src - 1);
  t.s1 = min(max(s + 1, 0), src - 1);
  t.w0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f));
  t.w1 = __float2int_rn(__fmul_rn(f, 2048.f));
  return t;
}

__device__ __forceinline__ int vlinear(int h0, int h1, int b0, int b1) {
  return (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;
}

__device__ __forceinline__ int sat_channel(float m0, float m1, float m2, float x0, float x1, float x2) {
  float v = __fmaf_rn(x2, m2, __fmaf_rn(x1, m1, __fmul_rn(x0, m0)));
  v = __fdiv_rn(v, 3.0f);
  v = fminf(fmaxf(v, 0.f), 255.f);
  return __float2int_rz(v);
}

// blockIdx.y = image.  out_w % 16 == 0 is required by the launcher (16-byte stores); rows are walked by a grid-stride
// loop over (row, 16-pixel group) pairs.  kNhwc: out is [B, H, W, 3] (a channels_last [B, 3, H, W] tensor), else
// [B, 3, H, W].
template <bool kNhwc>
__global__ void __launch_bounds__(256) image_pipeline_kernel(const mdseg_image_view* __restrict__ views,
                                                            const float* __restrict__ norm, int n_norm,
                                                            float* __restrict__ out, int out_h, int out_w) {
  __shared__ uint8_t s_lut[256];
  __shared__ float s_norm[3 * 256];
  const mdseg_image_view* vp = views + blockIdx.y;
  s_lut[threadIdx.x] = vp->lut[threadIdx.x];
  const int nrow = (vp->norm >= 0 && vp->norm < n_norm) ? vp->norm : 0;
  for (int i = threadIdx.x; i < 3 * 256; i += blockDim.x) s_norm[i] = norm[(int64_t)nrow * 768 + i];
  const uint8_t* src = vp->src;
  const int64_t rs = vp->src_row_stride;
  const int src_h = vp->src_h, src_w = vp->src_w, im_h = vp->im_h, im_w = vp->im_w;
  const int oy = vp->crop_y - vp->pad_top, ox = vp->crop_x - vp->pad_left, flip = vp->flip;
  const int c0 = vp->swap_rb ? 2 : 0, c2 = 2 - c0;  // source channel of output channel 0 / 2
  const int saturate = vp->saturate;
  const float md = vp->sat_diag, mo = vp->sat_off;
  __syncthreads();
  // OpenCV: inv_scale = (double)dsize / ssize; scale = 1. / inv_scale  (resize.cpp)
  const double scale_x = 1.0 / ((double)im_w / (double)src_w);
  const double scale_y = 1.0 / ((double)im_h / (double)src_h);
  const int groups = out_w / kPx;
  const int64_t total = (int64_t)out_h * groups;
  const int64_t plane = (int64_t)out_h * out_w;
  float* outb = out + (int64_t)blockIdx.y * 3 * plane;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int y = (int)(t / groups), x0 = (int)(t - (int64_t)y * groups) * kPx;
    const int Y = y + oy;
    const bool row_in = Y >= 0 && Y < im_h;
    Taps ty{0, 0, 0, 0};
    if (row_in) ty = linear_taps(Y, scale_y, src_h, false);
    const uint8_t* r0 = src + (int64_t)ty.s0 * rs;
    const uint8_t* r1 = src + (int64_t)ty.s1 * rs;
    float val[3][kPx];
#pragma unroll
    for (int i = 0; i < kPx; ++i) {
      const int xo = x0 + i;
      const int X = (flip ? out_w - 1 - xo : xo) + ox;
      int px[3] = {0, 0, 0};  // resized RGB, (0, 0, 0) in the padding
      if (row_in && X >= 0 && X < im_w) {
        const Taps tx = linear_taps(X, scale_x, src_w, true);
        const uint8_t* p00 = r0 + 3 * tx.s0;
        const uint8_t* p01 = r0 + 3 * tx.s1;
        const uint8_t* p10 = r1 + 3 * tx.s0;
        const uint8_t* p11 = r1 + 3 * tx.s1;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int sc = c == 0 ? c0 : (c == 1 ? 1 : c2);
          const int h0 = (int)__ldg(p00 + sc) * tx.w0 + (int)__ldg(p01 + sc) * tx.w1;
          const int h1 = (int)__ldg(p10 + sc) * tx.w0 + (int)__ldg(p11 + sc) * tx.w1;
          px[c] = vlinear(h0, h1, ty.w0, ty.w1);
        }
      }
      int q0 = s_lut[px[0]], q1 = s_lut[px[1]], q2 = s_lut[px[2]];
      if (saturate) {
        const float x0f = (float)q0, x1f = (float)q1, x2f = (float)q2;
        q0 = sat_channel(md, mo, mo, x0f, x1f, x2f);
        q1 = sat_channel(mo, md, mo, x0f, x1f, x2f);
        q2 = sat_channel(mo, mo, md, x0f, x1f, x2f);
      }
      val[0][i] = s_norm[q0];
      val[1][i] = s_norm[256 + q1];
      val[2][i] = s_norm[512 + q2];
    }
    if (kNhwc) {
      // 16 pixels x 3 channels = 192 contiguous bytes = twelve 16-byte stores
      float4* o = reinterpret_cast<float4*>(outb + ((int64_t)y * out_w + x0) * 3);
#pragma unroll
      for (int j = 0; j < 12; ++j) {
        float w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) w[k] = val[(4 * j + k) % 3][(4 * j + k) / 3];
        o[j] = make_float4(w[0], w[1], w[2], w[3]);
      }
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float4* o = reinterpret_cast<float4*>(outb + c * plane + (int64_t)y * out_w + x0);
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = make_float4(val[c][4 * j], val[c][4 * j + 1], val[c][4 * j + 2], val[c][4 * j + 3]);
      }
    }
  }
}

}  // namespace
}  // namespace mdseg

extern "C" int mdseg_image_pipeline(const mdseg_image_view* views, int n_images, const float* norm, int n_norm,
                                    float* out, int out_layout, int out_h, int out_w, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(views && out && n_images >= 0 && out_h > 0 && out_w > 0, "mdseg_image_pipeline: bad arguments");
  MDSEG_REQUIRE(out_w % kPx == 0, "mdseg_image_pipeline: out_w (%d) must be a multiple of 16", out_w);
  MDSEG_REQUIRE(norm && n_norm > 0, "mdseg_image_pipeline: at least one [3][256] normalisation table is required");
  MDSEG_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "mdseg_image_pipeline: out must be 16-byte aligned");
  if (n_images == 0) return 0;
  const int64_t threads = (int64_t)out_h * (out_w / kPx);
  int64_t blocks = ceil_div64(threads, 256);
  const int64_t cap = ceil_div64((int64_t)sm_count() * 8, n_images);  // eight resident CTAs per SM over all images
  if (blocks > cap) blocks = cap;
  const dim3 grid((unsigned)blocks, (unsigned)n_images);
  cudaStream_t s = (cudaStream_t)stream;
  switch (out_layout) {
    case MDSEG_NCHW:
      image_pipeline_kernel<false><<<grid, 256, 0, s>>>(views, norm, n_norm, out, out_h, out_w);
      break;
    case MDSEG_NHWC:
      image_pipeline_kernel<true><<<grid, 256, 0, s>>>(views, norm, n_norm, out, out_h, out_w);
      break;
    default:
      set_error("mdseg_image_pipeline: output layout %d (MDSEG_NCHW or MDSEG_NHWC)", out_layout);
      return 2;
  }
  MDSEG_LAUNCH_OK();
  return 0;
}
