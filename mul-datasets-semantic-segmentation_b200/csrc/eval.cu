// eval.cu — evaluator tail on the device (SURVEY §8 rows a11, a12, 10b).
//
// Reference work replaced (evaluate.py:136-181, MscEvalV0_Contrast.__call__):
//   logits = F.interpolate(logits, size=label HxW, mode='bilinear', align_corners=True)   :149-151
//   probs += torch.softmax(logits, dim=1)                                                  :164
//   (flip) logits = torch.flip(net(flip(im)), dims=(3,)) ; interpolate ; probs += softmax  :165-171
//   preds = torch.argmax(probs, dim=1)                                                     :172
//   label = F.interpolate(label.float(), size=(lH,lW), mode='nearest').long()              :156-157
// The upsampled logits are never materialised: each label pixel interpolates its
// 4 low-res corners per class on the fly (two sweeps: online max/sum, then the
// normalised probabilities are accumulated into `probs`).  The dominant traffic
// is the read-modify-write of probs (8*C bytes per pixel and pass).
#include <float.h>

#include "common.cuh"

namespace mdseg {
namespace {

// One label pixel of one pass: its four low-resolution corners (class 0) and interpolation weights.
template <typename T> struct EvalPixel {
  const T *q00, *q01, *q10, *q11;
  float l0h, l1h, l0w, l1w;
  __device__ __forceinline__ float at(int64_t o) const {
    return l0h * (l0w * to_f32<T>(q00[o]) + l1w * to_f32<T>(q01[o])) +
           l1h * (l0w * to_f32<T>(q10[o]) + l1w * to_f32<T>(q11[o]));
  }
};
constexpr int kEvBlk = 8;  // classes per block: 32 independent loads in flight per thread

// Soft-max statistics of a pixel: the running maximum is updated once per block of eight classes, so a block
// costs nine exponentials and its loads are independent.  Every evaluator kernel feeds the classes through these
// two functions in the same order (blocks of eight from class 0 while they fit, then single classes), which is
// what makes their sums bit-identical.
__device__ __forceinline__ void stats_feed8(const float (&z)[kEvBlk], float& m, float& sum) {
  float mb = z[0];
#pragma unroll
  for (int i = 1; i < kEvBlk; ++i) mb = fmaxf(mb, z[i]);
  const float mn = fmaxf(m, mb);
  float part = 0.f;
#pragma unroll
  for (int i = 0; i < kEvBlk; ++i) part += ex2_approx((z[i] - mn) * kLog2e);
  sum = fmaf(sum, ex2_approx((m - mn) * kLog2e), part);
  m = mn;
}
__device__ __forceinline__ void stats_feed1(float z, float& m, float& sum) {
  const float mn = fmaxf(m, z);
  sum = fmaf(sum, ex2_approx((m - mn) * kLog2e), ex2_approx((z - mn) * kLog2e));
  m = mn;
}
// probability of one class given the pixel's statistics, added to an accumulator (the subtraction is exact for
// nearby values, which a fused z * log2e - max * log2e would not be)
__device__ __forceinline__ float eval_add_prob(float acc, float z, float m, float inv) {
  return fmaf(ex2_approx((z - m) * kLog2e), inv, acc);
}
template <typename T>
__device__ __forceinline__ void eval_softmax_stats(const EvalPixel<T>& px, int C, int64_t hw, float& m, float& inv) {
  m = -FLT_MAX;
  float sum = 0.f;
  int c = 0;
  for (; c + kEvBlk <= C; c += kEvBlk) {
    float z[kEvBlk];
#pragma unroll
    for (int i = 0; i < kEvBlk; ++i) z[i] = px.at((int64_t)(c + i) * hw);
    stats_feed8(z, m, sum);
  }
  for (; c < C; ++c) stats_feed1(px.at((int64_t)c * hw), m, sum);
  inv = 1.0f / sum;
}

template <typename T>
__global__ void __launch_bounds__(256)
eval_accum_kernel(const T* __restrict__ logits, int C, int h, int w, float* __restrict__ probs, int H, int W,
                  AxisMap ym, AxisMap xm, int flip, int first) {
  const int64_t HW = (int64_t)H * W, hw = (int64_t)h * w;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < HW; p += (int64_t)gridDim.x * blockDim.x) {
    const int Y = (int)(p / W), X = (int)(p - (int64_t)Y * W);
    int y0, y1, x0, x1;
    float l0h, l1h, l0w, l1w;
    ym.at(Y, y0, y1, l0h, l1h);
    xm.at(X, x0, x1, l0w, l1w);
    if (flip) { x0 = w - 1 - x0; x1 = w - 1 - x1; }  // torch.flip(logits, dims=(3,)) before interpolate
    EvalPixel<T> px;
    px.q00 = logits + (int64_t)y0 * w + x0; px.q01 = logits + (int64_t)y0 * w + x1;
    px.q10 = logits + (int64_t)y1 * w + x0; px.q11 = logits + (int64_t)y1 * w + x1;
    px.l0h = l0h; px.l1h = l1h; px.l0w = l0w; px.l1w = l1w;
    float m, inv;
    eval_softmax_stats<T>(px, C, hw, m, inv);
    int c = 0;
    for (; c + kEvBlk <= C; c += kEvBlk) {
      float z[kEvBlk];
#pragma unroll
      for (int i = 0; i < kEvBlk; ++i) z[i] = px.at((int64_t)(c + i) * hw);
      float acc[kEvBlk];
#pragma unroll
      for (int i = 0; i < kEvBlk; ++i) acc[i] = first ? 0.f : probs[(int64_t)(c + i) * HW + p];
#pragma unroll
      for (int i = 0; i < kEvBlk; ++i) probs[(int64_t)(c + i) * HW + p] = eval_add_prob(acc[i], z[i], m, inv);
    }
    for (; c < C; ++c) {
      float* dst = probs + (int64_t)c * HW + p;
      *dst = eval_add_prob(first ? 0.f : *dst, px.at((int64_t)c * hw), m, inv);
    }
  }
}

template <typename L, bool kSmem>
__global__ void __launch_bounds__(256)
argmax_hist_kernel(const float* __restrict__ probs, int C, int64_t n_px, long long* __restrict__ pred,
                   const L* __restrict__ label, const uint8_t* __restrict__ lut, unsigned long long* __restrict__ hist,
                   int ignore, int* err_flag) {
  extern __shared__ unsigned sh_hist[];
  __shared__ uint8_t s_lut[256];
  const int bins = C * C;
  if (lut) s_lut[threadIdx.x] = lut[threadIdx.x];
  if (kSmem && hist)
    for (int i = threadIdx.x; i < bins; i += blockDim.x) sh_hist[i] = 0u;
  __syncthreads();
  int err = 0;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_px; p += (int64_t)gridDim.x * blockDim.x) {
    float best = probs[p];
    int arg = 0;
    for (int c = 1; c < C; ++c) {
      const float v = probs[(int64_t)c * n_px + p];
      if (v > best) { best = v; arg = c; }
    }
    if (pred) pred[p] = arg;
    if (hist) {
      int l = load_label<L>(label, p);
      if (lut) l = ((unsigned)l < 256u) ? (int)s_lut[l] : -1;
      if (l != ignore) {
        if ((unsigned)l >= (unsigned)C) err |= MDSEG_ERR_LABEL_RANGE;
        else if (kSmem) atomicAdd(&sh_hist[l * C + arg], 1u);
        else atomicAdd(&hist[l * C + arg], 1ull);
      }
    }
  }
  if (err && err_flag) atomicOr(err_flag, err);
  if (kSmem && hist) {
    __syncthreads();
    for (int i = threadIdx.x; i < bins; i += blockDim.x)
      if (sh_hist[i]) atomicAdd(&hist[i], (unsigned long long)sh_hist[i]);
  }
}

// ---- all (scale, flip) passes of one image without a probability tensor (SURVEY §8 f1) ------------------------
// The reference (and mdseg_eval_accum) read-modify-write a [C, H, W] fp32 probability tensor once per pass
// (1.26 GB for ADE at 1024 x 2048, 12 passes, 30 GB of traffic per image).  Here:
//   1. eval_stats_kernel: per pass and label pixel the soft-max statistics (max, 1 / sum) — 8 bytes;
//   2. eval_fused_kernel: a thread owns a label pixel and walks the classes in blocks of 16 whose accumulators
//      P[16] live in REGISTERS: for every pass it interpolates the block's logits on the fly and adds
//      ex2(z - max) / sum in pass order, then folds the block into the running arg-max; finally the confusion
//      matrix is updated.  The arithmetic and its order are those of eval_accum_kernel + argmax_hist_kernel, so
//      both routes give bit-identical predictions.
// Threads are tiled 16 x 16 over the label image so that a CTA's corner loads of one class cover a compact
// low-resolution patch (the re-reads stay in L1 / L2).  HBM sees the logits, the statistics, label and prediction.
constexpr int kEvTile = 16, kEvThreads = kEvTile * kEvTile;
constexpr int kEvCB = 16;  // classes per register block

struct EvalPassDev {
  const void* logits;
  AxisMap ym, xm;
  int h, w, flip;
};
struct EvalPassesDev {
  EvalPassDev p[MDSEG_MAX_EVAL_PASSES];
  int n;
};

template <typename T>
__device__ __forceinline__ EvalPixel<T> eval_pixel(const EvalPassDev& ep, int Y, int X) {
  int y0, y1, x0, x1;
  EvalPixel<T> px;
  ep.ym.at(Y, y0, y1, px.l0h, px.l1h);
  ep.xm.at(X, x0, x1, px.l0w, px.l1w);
  if (ep.flip) { x0 = ep.w - 1 - x0; x1 = ep.w - 1 - x1; }  // torch.flip(logits, dims=(3,)) before interpolate
  const T* base = (const T*)ep.logits;
  px.q00 = base + (int64_t)y0 * ep.w + x0; px.q01 = base + (int64_t)y0 * ep.w + x1;
  px.q10 = base + (int64_t)y1 * ep.w + x0; px.q11 = base + (int64_t)y1 * ep.w + x1;
  return px;
}

template <typename T>
__global__ void __launch_bounds__(kEvThreads)
eval_stats_kernel(const __grid_constant__ EvalPassesDev ps, int C, int H, int W, float2* __restrict__ stats) {
  const int Y = blockIdx.y * kEvTile + (threadIdx.x >> 4), X = blockIdx.x * kEvTile + (threadIdx.x & 15);
  if (Y >= H || X >= W) return;
  const int s = blockIdx.z;
  const EvalPassDev& ep = ps.p[s];
  const EvalPixel<T> px = eval_pixel<T>(ep, Y, X);
  float m, inv;
  eval_softmax_stats<T>(px, C, (int64_t)ep.h * ep.w, m, inv);
  stats[((int64_t)s * H + Y) * W + X] = make_float2(m, inv);
}

template <typename T, typename L>
__global__ void __launch_bounds__(kEvThreads)
eval_fused_kernel(const __grid_constant__ EvalPassesDev ps, int C, int H, int W, const float2* __restrict__ stats,
                  long long* __restrict__ pred, const L* __restrict__ label, const uint8_t* __restrict__ lut,
                  unsigned long long* __restrict__ hist, int ignore, int* err_flag) {
  const int Y = blockIdx.y * kEvTile + (threadIdx.x >> 4), X = blockIdx.x * kEvTile + (threadIdx.x & 15);
  if (Y >= H || X >= W) return;
  const int64_t p = (int64_t)Y * W + X, HW = (int64_t)H * W;
  float best = -FLT_MAX;
  int arg = 0;
  for (int c0 = 0; c0 < C; c0 += kEvCB) {
    float P[kEvCB];
#pragma unroll
    for (int i = 0; i < kEvCB; ++i) P[i] = 0.f;
    const int nc = (C - c0) < kEvCB ? (C - c0) : kEvCB;
    for (int s = 0; s < ps.n; ++s) {
      const EvalPassDev& ep = ps.p[s];
      const EvalPixel<T> px = eval_pixel<T>(ep, Y, X);
      const int64_t hw = (int64_t)ep.h * ep.w;
      const float2 st = stats[(int64_t)s * HW + p];
      if (nc == kEvCB) {
        float z[kEvCB];
#pragma unroll
        for (int i = 0; i < kEvCB; ++i) z[i] = px.at((int64_t)(c0 + i) * hw);
#pragma unroll
        for (int i = 0; i < kEvCB; ++i) P[i] = eval_add_prob(P[i], z[i], st.x, st.y);
      } else {
#pragma unroll
        for (int i = 0; i < kEvCB; ++i)
          if (i < nc) P[i] = eval_add_prob(P[i], px.at((int64_t)(c0 + i) * hw), st.x, st.y);
      }
    }
#pragma unroll
    for (int i = 0; i < kEvCB; ++i)
      if (i < nc && (P[i] > best || (c0 + i) == 0)) { best = P[i]; arg = c0 + i; }
  }
  if (pred) pred[p] = arg;
  if (hist) {
    int l = load_label<L>(label, p);
    if (lut) l = ((unsigned)l < 256u) ? (int)__ldg(lut + l) : -1;
    if (l != ignore) {
      if ((unsigned)l >= (unsigned)C) { if (err_flag) atomicOr(err_flag, MDSEG_ERR_LABEL_RANGE); }
      else atomicAdd(&hist[(int64_t)l * C + arg], 1ull);
    }
  }
}

// ---- the same two kernels with the low-resolution patch of a tile staged in shared memory -------------------
// For passes that do not down-sample (h <= H, w <= W) the 16 x 16 label tile of a CTA interpolates inside a
// patch of at most 17 x 17 logits per class.  The direct kernels fetch each corner from L1 / L2 (four lookups per
// pixel, class and pass — the L1 tag stage is what binds them); here the CTA copies the patch of 16 classes once
// (one or two elements per thread and class, double-buffered, one barrier per block) and the corners come from
// shared memory, mostly as broadcasts.
constexpr int kEvPatch = 18;
constexpr int kEvPatchElems = kEvPatch * kEvPatch;

struct EvalPatch {
  int o00, o01, o10, o11;      // this thread's corners inside the patch of one class
  float l0h, l1h, l0w, l1w;
  int e[2];                    // patch elements this thread copies (-1: none) ...
  int64_t src[2];              // ... and their offsets inside a class plane
  __device__ __forceinline__ float at(const float* pc) const {
    return l0h * (l0w * pc[o00] + l1w * pc[o01]) + l1h * (l0w * pc[o10] + l1w * pc[o11]);
  }
};

__device__ __forceinline__ EvalPatch eval_patch(const EvalPassDev& ep, int Y, int X, int H, int W) {
  const int Yt0 = blockIdx.y * kEvTile, Xt0 = blockIdx.x * kEvTile;
  const int Yl = min(Yt0 + kEvTile - 1, H - 1), Xl = min(Xt0 + kEvTile - 1, W - 1);
  const int r0 = ep.ym.floor_at(Yt0), r1 = min(ep.h - 1, ep.ym.floor_at(Yl) + 1);
  const int c0 = ep.xm.floor_at(Xt0), c1 = min(ep.w - 1, ep.xm.floor_at(Xl) + 1);
  const int n_rows = r1 - r0 + 1, n_cols = c1 - c0 + 1;
  EvalPatch g;
  int y0, y1, x0, x1;
  ep.ym.at(Y, y0, y1, g.l0h, g.l1h);
  ep.xm.at(X, x0, x1, g.l0w, g.l1w);
  g.o00 = (y0 - r0) * n_cols + (x0 - c0); g.o01 = (y0 - r0) * n_cols + (x1 - c0);
  g.o10 = (y1 - r0) * n_cols + (x0 - c0); g.o11 = (y1 - r0) * n_cols + (x1 - c0);
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int e = threadIdx.x + k * kEvThreads;
    g.e[k] = -1;
    g.src[k] = 0;
    if (e < n_rows * n_cols) {
      const int ry = e / n_cols, rx = e - ry * n_cols;
      const int sx = ep.flip ? ep.w - 1 - (c0 + rx) : c0 + rx;  // torch.flip(logits, dims=(3,)) before interpolate
      g.e[k] = e;
      g.src[k] = (int64_t)(r0 + ry) * ep.w + sx;
    }
  }
  return g;
}

// copy the patch of classes [c0, c0 + nc) of one pass into `buf` ([kEvCB][kEvPatchElems])
template <typename T>
__device__ __forceinline__ void eval_stage(const EvalPassDev& ep, const EvalPatch& g, int c0, int nc, float* buf) {
  const T* base = (const T*)ep.logits + (int64_t)c0 * ep.h * ep.w;
  const int64_t hw = (int64_t)ep.h * ep.w;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    if (g.e[k] >= 0) {
      float v[kEvCB];
#pragma unroll
      for (int i = 0; i < kEvCB; ++i) v[i] = (i < nc) ? to_f32<T>(base[(int64_t)i * hw + g.src[k]]) : 0.f;
#pragma unroll
      for (int i = 0; i < kEvCB; ++i) buf[i * kEvPatchElems + g.e[k]] = v[i];
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(kEvThreads)
eval_stats_staged_kernel(const __grid_constant__ EvalPassesDev ps, int C, int H, int W, float2* __restrict__ stats) {
  __shared__ float patch[2][kEvCB * kEvPatchElems];
  const int Yr = blockIdx.y * kEvTile + (threadIdx.x >> 4), Xr = blockIdx.x * kEvTile + (threadIdx.x & 15);
  const bool inside = Yr < H && Xr < W;
  const int Y = min(Yr, H - 1), X = min(Xr, W - 1);  // threads outside the image still help with the copies
  const int s = blockIdx.z;
  const EvalPassDev& ep = ps.p[s];
  const EvalPatch g = eval_patch(ep, Y, X, H, W);
  float m = -FLT_MAX, sum = 0.f;
  int it = 0;
  for (int c0 = 0; c0 < C; c0 += kEvCB, ++it) {
    const int nc = (C - c0) < kEvCB ? (C - c0) : kEvCB;
    float* buf = patch[it & 1];
    eval_stage<T>(ep, g, c0, nc, buf);
    __syncthreads();
#pragma unroll
    for (int hb = 0; hb < kEvCB / kEvBlk; ++hb) {
      const int cb = c0 + hb * kEvBlk;
      if (cb + kEvBlk <= C) {
        float z[kEvBlk];
#pragma unroll
        for (int i = 0; i < kEvBlk; ++i) z[i] = g.at(buf + (hb * kEvBlk + i) * kEvPatchElems);
        stats_feed8(z, m, sum);
      } else {
        for (int c = cb; c < C && c < cb + kEvBlk; ++c) stats_feed1(g.at(buf + (c - c0) * kEvPatchElems), m, sum);
      }
    }
  }
  if (inside) stats[((int64_t)s * H + Y) * W + X] = make_float2(m, 1.0f / sum);
}

template <typename T, typename L>
__global__ void __launch_bounds__(kEvThreads)
eval_fused_staged_kernel(const __grid_constant__ EvalPassesDev ps, int C, int H, int W,
                         const float2* __restrict__ stats, long long* __restrict__ pred, const L* __restrict__ label,
                         const uint8_t* __restrict__ lut, unsigned long long* __restrict__ hist, int ignore,
                         int* err_flag) {
  __shared__ float patch[2][kEvCB * kEvPatchElems];
  const int Yr = blockIdx.y * kEvTile + (threadIdx.x >> 4), Xr = blockIdx.x * kEvTile + (threadIdx.x & 15);
  const bool inside = Yr < H && Xr < W;
  const int Y = min(Yr, H - 1), X = min(Xr, W - 1);
  const int64_t p = (int64_t)Y * W + X, HW = (int64_t)H * W;
  float best = -FLT_MAX;
  int arg = 0, it = 0;
  for (int c0 = 0; c0 < C; c0 += kEvCB) {
    float P[kEvCB];
#pragma unroll
    for (int i = 0; i < kEvCB; ++i) P[i] = 0.f;
    const int nc = (C - c0) < kEvCB ? (C - c0) : kEvCB;
    for (int s = 0; s < ps.n; ++s, ++it) {
      const EvalPassDev& ep = ps.p[s];
      const EvalPatch g = eval_patch(ep, Y, X, H, W);
      float* buf = patch[it & 1];
      eval_stage<T>(ep, g, c0, nc, buf);
      const float2 st = stats[(int64_t)s * HW + p];
      __syncthreads();
#pragma unroll
      for (int i = 0; i < kEvCB; ++i)
        if (i < nc) P[i] = eval_add_prob(P[i], g.at(buf + i * kEvPatchElems), st.x, st.y);
    }
#pragma unroll
    for (int i = 0; i < kEvCB; ++i)
      if (i < nc && (P[i] > best || (c0 + i) == 0)) { best = P[i]; arg = c0 + i; }
  }
  if (!inside) return;
  if (pred) pred[p] = arg;
  if (hist) {
    int l = load_label<L>(label, p);
    if (lut) l = ((unsigned)l < 256u) ? (int)__ldg(lut + l) : -1;
    if (l != ignore) {
      if ((unsigned)l >= (unsigned)C) { if (err_flag) atomicOr(err_flag, MDSEG_ERR_LABEL_RANGE); }
      else atomicAdd(&hist[(int64_t)l * C + arg], 1ull);
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
label_nearest_kernel(const T* __restrict__ in, int Hin, int Win, T* __restrict__ out, int Hout, int Wout, int n,
                     float sy, float sx) {
  const int64_t total = (int64_t)n * Hout * Wout;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int xo = (int)(i % Wout);
    const int64_t r = i / Wout;
    const int yo = (int)(r % Hout);
    const int64_t b = r / Hout;
    // ATen nearest_neighbor_compute_source_index: min(floor(dst * scale), in - 1)
    int ys = (int)floorf((float)yo * sy);
    int xs = (int)floorf((float)xo * sx);
    ys = ys > Hin - 1 ? Hin - 1 : ys;
    xs = xs > Win - 1 ? Win - 1 : xs;
    out[i] = in[(b * Hin + ys) * Win + xs];
  }
}

int grid_for(int64_t n) {
  int64_t blocks = ceil_div64(n > 0 ? n : 1, 256);
  int64_t cap = (int64_t)sm_count() * 8;
  return (int)(blocks > cap ? cap : blocks);
}

template <typename L>
int launch_argmax(const float* probs, int C, int64_t n_px, int64_t* pred, const void* label, const uint8_t* lut,
                  int64_t* hist, int ignore, int32_t* ef, cudaStream_t s) {
  const size_t smem = (size_t)C * C * 4;
  const bool use_smem = hist && smem <= 96 * 1024;
  if (use_smem) {
    auto k = argmax_hist_kernel<L, true>;
    if (smem > 48 * 1024) MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int blocks = grid_for(n_px);
    int cap = sm_count() * (smem > 24 * 1024 ? 2 : 8);
    if (blocks > cap) blocks = cap;
    k<<<blocks, 256, smem, s>>>(probs, C, n_px, (long long*)pred, (const L*)label, lut, (unsigned long long*)hist,
                                ignore, ef);
  } else {
    argmax_hist_kernel<L, false><<<grid_for(n_px), 256, 0, s>>>(probs, C, n_px, (long long*)pred, (const L*)label,
                                                                lut, (unsigned long long*)hist, ignore, ef);
  }
  MDSEG_LAUNCH_OK();
  return 0;
}

}  // namespace
}  // namespace mdseg

extern "C" int mdseg_eval_accum(const void* logits, int dtype, int C, int h, int w, float* probs, int H, int W,
                                int flip, int first, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(logits && probs && C > 0 && h > 0 && w > 0 && H > 0 && W > 0, "mdseg_eval_accum: bad arguments");
  AxisMap ym{axis_scale(h, H), h}, xm{axis_scale(w, W), w};
  cudaStream_t s = (cudaStream_t)stream;
  const int g = grid_for((int64_t)H * W);
  return with_float_type(dtype, "mdseg_eval_accum", "dtype", [&](auto t) {
    using T = typename decltype(t)::type;
    eval_accum_kernel<T><<<g, 256, 0, s>>>((const T*)logits, C, h, w, probs, H, W, ym, xm, flip, first);
    MDSEG_LAUNCH_OK();
    return 0;
  });
}

extern "C" int mdseg_argmax_hist(const float* probs, int C, int64_t n_px, int64_t* pred, const void* label,
                                 int label_dtype, const uint8_t* lut256, int64_t* hist, int ignore,
                                 int32_t* err_flag, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(probs && C > 0 && n_px >= 0, "mdseg_argmax_hist: bad arguments");
  MDSEG_REQUIRE(!hist || (label && err_flag), "mdseg_argmax_hist: hist needs label and err_flag");
  MDSEG_REQUIRE((int64_t)C * C < (1LL << 31), "mdseg_argmax_hist: C too large");
  if (n_px == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (!hist) return launch_argmax<uint8_t>(probs, C, n_px, pred, nullptr, nullptr, nullptr, ignore, err_flag, s);
  return with_int_type(label_dtype, "mdseg_argmax_hist", "label dtype", [&](auto l) {
    return launch_argmax<typename decltype(l)::type>(probs, C, n_px, pred, label, lut256, hist, ignore, err_flag, s);
  });
}

extern "C" int mdseg_label_nearest(const void* in, int dtype, int Hin, int Win, void* out, int Hout, int Wout,
                                   int n_images, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(in && out && Hin > 0 && Win > 0 && Hout > 0 && Wout > 0 && n_images >= 0,
                "mdseg_label_nearest: bad arguments");
  if (n_images == 0) return 0;
  const float sy = (float)Hin / (float)Hout, sx = (float)Win / (float)Wout;
  const int g = grid_for((int64_t)n_images * Hout * Wout);
  cudaStream_t s = (cudaStream_t)stream;
  return with_int_type(dtype, "mdseg_label_nearest", "dtype", [&](auto l) {
    using L = typename decltype(l)::type;
    label_nearest_kernel<L><<<g, 256, 0, s>>>((const L*)in, Hin, Win, (L*)out, Hout, Wout, n_images, sy, sx);
    MDSEG_LAUNCH_OK();
    return 0;
  });
}

namespace mdseg {
namespace {
template <typename T>
int launch_eval_fused(const EvalPassesDev& ps, int C, int H, int W, float2* stats, int64_t* pred, const void* label,
                      int label_dtype, const uint8_t* lut, int64_t* hist, int ignore, int32_t* ef, cudaStream_t s) {
  const dim3 grid((unsigned)((W + kEvTile - 1) / kEvTile), (unsigned)((H + kEvTile - 1) / kEvTile));
  bool staged = true;  // every pass up-samples: a tile's patch has at most 17 x 17 logits per class
  for (int i = 0; i < ps.n; ++i) staged = staged && ps.p[i].h <= H && ps.p[i].w <= W;
  if (staged) eval_stats_staged_kernel<T><<<dim3(grid.x, grid.y, (unsigned)ps.n), kEvThreads, 0, s>>>(ps, C, H, W, stats);
  else eval_stats_kernel<T><<<dim3(grid.x, grid.y, (unsigned)ps.n), kEvThreads, 0, s>>>(ps, C, H, W, stats);
  MDSEG_LAUNCH_OK();
  return with_int_type(hist ? label_dtype : MDSEG_U8, "mdseg_eval_fused", "label dtype", [&](auto l) {
    using L = typename decltype(l)::type;
    if (staged)
      eval_fused_staged_kernel<T, L><<<grid, kEvThreads, 0, s>>>(ps, C, H, W, stats, (long long*)pred, (const L*)label,
                                                                 lut, (unsigned long long*)hist, ignore, ef);
    else
      eval_fused_kernel<T, L><<<grid, kEvThreads, 0, s>>>(ps, C, H, W, stats, (long long*)pred, (const L*)label, lut,
                                                          (unsigned long long*)hist, ignore, ef);
    MDSEG_LAUNCH_OK();
    return 0;
  });
}
}  // namespace
}  // namespace mdseg

extern "C" size_t mdseg_eval_fused_workspace_bytes(int n_passes, int H, int W) {
  if (n_passes <= 0 || H <= 0 || W <= 0) return 256;
  return (size_t)n_passes * H * W * 8 + 256;
}

extern "C" int mdseg_eval_fused(const mdseg_eval_passes* passes, int C, int H, int W, int64_t* pred, const void* label,
                                int label_dtype, const uint8_t* lut256, int64_t* hist, int ignore, void* workspace,
                                size_t workspace_bytes, int32_t* err_flag, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(passes && passes->n_passes > 0 && passes->n_passes <= MDSEG_MAX_EVAL_PASSES,
                "mdseg_eval_fused: 1..%d passes", MDSEG_MAX_EVAL_PASSES);
  MDSEG_REQUIRE(C > 0 && H > 0 && W > 0 && H <= 65535 * kEvTile && (int64_t)C * C < (1LL << 31),
                "mdseg_eval_fused: bad shape");
  MDSEG_REQUIRE(pred || hist, "mdseg_eval_fused: nothing to compute (pred and hist are NULL)");
  MDSEG_REQUIRE(!hist || (label && err_flag), "mdseg_eval_fused: hist needs label and err_flag");
  MDSEG_REQUIRE(is_float_dtype(passes->dtype), "mdseg_eval_fused: unsupported dtype %d", passes->dtype);
  MDSEG_REQUIRE(workspace && workspace_bytes >= mdseg_eval_fused_workspace_bytes(passes->n_passes, H, W),
                "mdseg_eval_fused: workspace too small");
  EvalPassesDev ps;
  ps.n = passes->n_passes;
  for (int i = 0; i < ps.n; ++i) {
    const mdseg_eval_pass& e = passes->p[i];
    MDSEG_REQUIRE(e.logits && e.h > 0 && e.w > 0, "mdseg_eval_fused: bad pass %d", i);
    ps.p[i].logits = e.logits;
    ps.p[i].ym = AxisMap{axis_scale(e.h, H), e.h};
    ps.p[i].xm = AxisMap{axis_scale(e.w, W), e.w};
    ps.p[i].h = e.h; ps.p[i].w = e.w; ps.p[i].flip = e.flip;
  }
  float2* stats = reinterpret_cast<float2*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  cudaStream_t s = (cudaStream_t)stream;
  return with_float_type(passes->dtype, "mdseg_eval_fused", "dtype", [&](auto t) {
    return launch_eval_fused<typename decltype(t)::type>(ps, C, H, W, stats, pred, label, label_dtype, lut256, hist,
                                                         ignore, err_flag, s);
  });
}
