// ohem_ce.cu — full-resolution per-pixel cross-entropy forward / backward
// (SURVEY §8 rows a7, a9; first half of a8).
//
// Reference work replaced (lib/loss/ohem_ce_loss.py:19,25-30 and the autograd
// replay of :34):
//   loss = CrossEntropyLoss(ignore_index=255, reduction='none')(logits, labels).view(-1)
//   n_min = labels[labels != 255].numel() // 16 ; loss_hard = loss[loss > thresh]
// ATen runs log_softmax (materialising a second [N,C,H,W]) + nll_loss2d +
// compare + nonzero + index; here the logits are read ONCE: each thread owns
// 4 (fp32) or 8 (bf16/fp16) consecutive pixels along W, streams the C channel
// planes with 128-bit loads (8 in flight), keeps a chunked online
// log-sum-exp in registers, and writes loss + lse (8 B/px).  The three OHEM
// counters are reduced warp -> CTA -> one 64-bit atomic each.
// Backward re-reads the logits only for vectors that contain a selected pixel.
//
// Algorithmic bytes per pixel (fwd + bwd): 3*C*e + 2*L + 16 (+4 in select).
#include <float.h>

#include "tma_util.cuh"

namespace mdseg {
namespace {

constexpr int kKC = 8;  // channel planes in flight per thread

// ---- selection predicate shared by every backward kernel -------------------
struct SelParams {
  float thresh, kth, w;  // w = grad_out * scale / |S|
  unsigned mode;
};
__device__ __forceinline__ SelParams load_sel(const mdseg_ohem_state* st, const float* grad_out, float grad_scale) {
  SelParams p;
  p.thresh = st->thresh;
  p.kth = st->kth;
  p.mode = st->mode;
  float g = grad_out ? grad_out[0] : 1.0f;
  p.w = g * grad_scale * st->inv_n_sel;
  return p;
}
// Membership in S is a pure function of the stored loss: in top-k mode
// mdseg_ohem_select has already demoted the ties that did not make the quota
// to just below kth, so `loss >= kth` is exact.
__device__ __forceinline__ bool is_selected(const SelParams& p, float loss) {
  return p.mode == 0 ? (loss > p.thresh) : (loss >= p.kth);
}

template <int PX> __device__ __forceinline__ void store_f32(float* p, const float (&v)[PX]) {
  if constexpr (PX == 1) {
    p[0] = v[0];
  } else {
#pragma unroll
    for (int j = 0; j < PX; j += 4)
      stg_stream_v4(p + j, make_int4(__float_as_int(v[j]), __float_as_int(v[j + 1]), __float_as_int(v[j + 2]),
                                     __float_as_int(v[j + 3])));
  }
}

// ---- NCHW forward ------------------------------------------------------------
template <typename T, typename L, int PX>
__global__ void __launch_bounds__(256)
ce_fwd_nchw_kernel(const T* __restrict__ logits, const L* __restrict__ labels, int N, int C, int64_t HW, int ignore,
                   float* __restrict__ loss_px, float* __restrict__ lse_px, mdseg_ohem_state* st, int* err_flag) {
  const int64_t groups_per_img = HW / PX;
  const int64_t n_groups = groups_per_img * N;
  const float thresh = st->thresh;
  unsigned n_valid = 0, n_hard = 0, n_px = 0;
  double sum_hard = 0.0;
  int err = 0;

  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = g / groups_per_img;
    const int64_t p0 = (g - n * groups_per_img) * PX;
    const T* base = logits + (n * C) * HW + p0;
    const int64_t px0 = n * HW + p0;

    int lab[PX];
#pragma unroll
    for (int i = 0; i < PX; ++i) lab[i] = load_label<L>(labels, px0 + i);

    float m[PX], s[PX], zl[PX];
#pragma unroll
    for (int i = 0; i < PX; ++i) { m[i] = -FLT_MAX; s[i] = 0.f; zl[i] = 0.f; }

    for (int c0 = 0; c0 < C; c0 += kKC) {
      float v[kKC][PX];
#pragma unroll
      for (int k = 0; k < kKC; ++k) {
        if (c0 + k < C) {
          VecLoad<T, PX>::load(base + (int64_t)(c0 + k) * HW, v[k]);
        } else {
#pragma unroll
          for (int i = 0; i < PX; ++i) v[k][i] = -FLT_MAX;
        }
      }
#pragma unroll
      for (int i = 0; i < PX; ++i) {
        float cm = v[0][i];
#pragma unroll
        for (int k = 1; k < kKC; ++k) cm = fmaxf(cm, v[k][i]);
        const float mn = fmaxf(m[i], cm);
        float acc = s[i] * ex2_approx((m[i] - mn) * kLog2e);
#pragma unroll
        for (int k = 0; k < kKC; ++k) {
          acc += ex2_approx((v[k][i] - mn) * kLog2e);
          zl[i] = (c0 + k == lab[i]) ? v[k][i] : zl[i];
        }
        s[i] = acc;
        m[i] = mn;
      }
    }

    float lo[PX], ls[PX];
#pragma unroll
    for (int i = 0; i < PX; ++i) {
      const float lse = m[i] + logf(s[i]);
      ls[i] = lse;
      const bool ign = lab[i] == ignore;
      const bool ok = (unsigned)lab[i] < (unsigned)C;
      if (!ign && !ok) err |= MDSEG_ERR_LABEL_RANGE;
      const float l = (ok && !ign) ? (lse - zl[i]) : 0.f;
      lo[i] = l;
      n_valid += (ok && !ign) ? 1u : 0u;
      if (l > thresh) { ++n_hard; sum_hard += (double)l; }
    }
    n_px += PX;
    store_f32<PX>(loss_px + px0, lo);
    store_f32<PX>(lse_px + px0, ls);
  }
  if (err) atomicOr(err_flag, err);
  block_accumulate_stats(st, n_valid, n_hard, sum_hard, n_px);
}

// ---- NCHW backward -------------------------------------------------------------
template <typename T, typename L, int PX>
__global__ void __launch_bounds__(256)
ce_bwd_nchw_kernel(const T* __restrict__ logits, const L* __restrict__ labels, int N, int C, int64_t HW, int ignore,
                   const float* __restrict__ loss_px, const float* __restrict__ lse_px, mdseg_ohem_state* st,
                   const float* __restrict__ grad_out, float grad_scale, T* __restrict__ dlogits) {
  const int64_t groups_per_img = HW / PX;
  const int64_t n_groups = groups_per_img * N;
  const SelParams sp = load_sel(st, grad_out, grad_scale);

  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = g / groups_per_img;
    const int64_t p0 = (g - n * groups_per_img) * PX;
    const int64_t px0 = n * HW + p0;
    const T* base = logits + (n * C) * HW + p0;
    T* dbase = dlogits + (n * C) * HW + p0;

    int lab[PX];
    float wgt[PX], lse2[PX];
    bool any = false;
#pragma unroll
    for (int i = 0; i < PX; ++i) {
      lab[i] = load_label<L>(labels, px0 + i);
      const float l = loss_px[px0 + i];
      const bool valid = (lab[i] != ignore) && ((unsigned)lab[i] < (unsigned)C);
      const bool sel = is_selected(sp, l) && valid;
      wgt[i] = sel ? sp.w : 0.f;
      lse2[i] = lse_px[px0 + i] * kLog2e;
      any |= sel;
    }
    if (!any) {
      float z[PX];
#pragma unroll
      for (int i = 0; i < PX; ++i) z[i] = 0.f;
      for (int c = 0; c < C; ++c) VecLoad<T, PX>::store(dbase + (int64_t)c * HW, z);
      continue;
    }
    for (int c0 = 0; c0 < C; c0 += kKC) {
      float v[kKC][PX];
#pragma unroll
      for (int k = 0; k < kKC; ++k)
        if (c0 + k < C) VecLoad<T, PX>::load(base + (int64_t)(c0 + k) * HW, v[k]);
#pragma unroll
      for (int k = 0; k < kKC; ++k) {
        if (c0 + k < C) {
          float d[PX];
#pragma unroll
          for (int i = 0; i < PX; ++i) {
            const float p = ex2_approx(fmaf(v[k][i], kLog2e, -lse2[i]));
            d[i] = wgt[i] * (p - ((c0 + k == lab[i]) ? 1.f : 0.f));
          }
          VecLoad<T, PX>::store(dbase + (int64_t)(c0 + k) * HW, d);
        }
      }
    }
  }
}

// ---- NHWC (channels_last): one warp per pixel, lanes stride the channels ------
template <typename T, typename L>
__global__ void __launch_bounds__(256)
ce_fwd_nhwc_kernel(const T* __restrict__ logits, const L* __restrict__ labels, int64_t P, int C, int ignore,
                   float* __restrict__ loss_px, float* __restrict__ lse_px, mdseg_ohem_state* st, int* err_flag) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const float thresh = st->thresh;
  unsigned n_valid = 0, n_hard = 0, n_px = 0;
  double sum_hard = 0.0;
  int err = 0;
  for (int64_t p = warp; p < P; p += n_warps) {
    const T* row = logits + p * C;
    float m = -FLT_MAX;
    for (int c = lane; c < C; c += 32) m = fmaxf(m, to_f32<T>(row[c]));
    m = warp_max(m);
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s += ex2_approx((to_f32<T>(row[c]) - m) * kLog2e);
    s = warp_sum(s);
    if (lane == 0) {
      const int lab = load_label<L>(labels, p);
      const float lse = m + logf(s);
      const bool ign = lab == ignore;
      const bool ok = (unsigned)lab < (unsigned)C;
      if (!ign && !ok) err |= MDSEG_ERR_LABEL_RANGE;
      const float l = (ok && !ign) ? (lse - to_f32<T>(row[lab])) : 0.f;
      loss_px[p] = l;
      lse_px[p] = lse;
      n_valid += (ok && !ign) ? 1u : 0u;
      if (l > thresh) { ++n_hard; sum_hard += (double)l; }
      ++n_px;
    }
  }
  if (err) atomicOr(err_flag, err);
  block_accumulate_stats(st, n_valid, n_hard, sum_hard, n_px);
}

template <typename T, typename L>
__global__ void __launch_bounds__(256)
ce_bwd_nhwc_kernel(const T* __restrict__ logits, const L* __restrict__ labels, int64_t P, int C, int ignore,
                   const float* __restrict__ loss_px, const float* __restrict__ lse_px, mdseg_ohem_state* st,
                   const float* __restrict__ grad_out, float grad_scale, T* __restrict__ dlogits) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const SelParams sp = load_sel(st, grad_out, grad_scale);
  for (int64_t p = warp; p < P; p += n_warps) {
    int lab = 0;
    float w = 0.f, lse2 = 0.f;
    if (lane == 0) {
      lab = load_label<L>(labels, p);
      const bool valid = (lab != ignore) && ((unsigned)lab < (unsigned)C);
      w = (is_selected(sp, loss_px[p]) && valid) ? sp.w : 0.f;
      lse2 = lse_px[p] * kLog2e;
    }
    lab = __shfl_sync(0xffffffffu, lab, 0);
    w = __shfl_sync(0xffffffffu, w, 0);
    lse2 = __shfl_sync(0xffffffffu, lse2, 0);
    const T* row = logits + p * C;
    T* drow = dlogits + p * C;
    if (w == 0.f) {
      for (int c = lane; c < C; c += 32) drow[c] = from_f32<T>(0.f);
    } else {
      for (int c = lane; c < C; c += 32) {
        const float pr = ex2_approx(fmaf(to_f32<T>(row[c]), kLog2e, -lse2));
        drow[c] = from_f32<T>(w * (pr - ((c == lab) ? 1.f : 0.f)));
      }
    }
  }
}


// ---- NHWC (channels_last), tiled: a tile of TP pixels x C channels is CONTIGUOUS in memory -----------------------
// One persistent 256-thread CTA per SM.  A tile arrives with a single cp.async.bulk (no thread copies anything) into
// one of two shared-memory stages while the previous tile is being computed; 256 / TP threads share a pixel and walk
// its channels interleaved (for even C in an order rotated by the pixel index, so that the row stride C does not map
// the pixels of a warp onto the same banks); the backward overwrites the tile in place and it leaves with one bulk
// store.  The label-class logit is one direct read instead of a compare per channel.
#ifndef MDSEG_TILE_THREADS
#define MDSEG_TILE_THREADS 1024
#endif
constexpr int kTileThreads = MDSEG_TILE_THREADS;
constexpr int kTileStageBytes = 100 * 1024;

// one tile of `bytes` global -> shared, completion on `bar`
__device__ __forceinline__ void tile_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  tma::mbar_expect_tx(bar, bytes);
  tma::bulk_g2s(dst, src, bytes, bar);
}

// pixels per tile for C channels of `esz` bytes, so that the tile fills (at most) one stage: a multiple of the CTA size
// (one or more pixels per thread) or, for wide rows, a power of two below it (2 .. 32 threads per pixel); 0 = no fit
int tile_pixels(int C, int esz) {
  const size_t fit = (size_t)kTileStageBytes / ((size_t)C * esz);
  if (fit >= (size_t)kTileThreads) return (int)(fit / kTileThreads > 4 ? 4 : fit / kTileThreads) * kTileThreads;
  int tp = kTileThreads / 2;
  while (tp >= 32 && (size_t)tp > fit) tp >>= 1;
  return tp >= 32 ? tp : 0;
}

template <typename T, typename L, bool BWD>
__global__ void __launch_bounds__(kTileThreads, 1)
ce_nhwc_tile_kernel(const T* __restrict__ logits, const L* __restrict__ labels, int64_t n_tiles, int TP, int C, int ignore,
                    float* __restrict__ loss_px, float* __restrict__ lse_px, mdseg_ohem_state* st, int* err_flag,
                    const float* __restrict__ grad_out, float grad_scale, T* __restrict__ dlogits) {
  extern __shared__ __align__(128) unsigned char tile_smem[];
  __shared__ __align__(8) uint64_t bars[2];
  const uint32_t tile_bytes = (uint32_t)TP * C * sizeof(T);
  const uint32_t stage_stride = (tile_bytes + 127u) & ~127u;
  const int tpc = TP >= kTileThreads ? 1 : kTileThreads / TP;  // threads per pixel: 1, 2, 4 or 8
  const int ppt = TP >= kTileThreads ? TP / kTileThreads : 1;  // pixels per thread: 1 .. 8
  const int part = threadIdx.x % tpc;
  const bool rotate = (C % 2) == 0;
  const float thresh = st->thresh;
  SelParams sp;
  if (BWD) sp = load_sel(st, grad_out, grad_scale);
  unsigned n_valid = 0, n_hard = 0, n_px = 0;
  double sum_hard = 0.0;
  int err = 0;

  if (threadIdx.x == 0) {
    tma::mbar_init(&bars[0], 1);
    tma::mbar_init(&bars[1], 1);
    tma::mbar_fence_init();
    if ((int64_t)blockIdx.x < n_tiles)
      tile_load(tile_smem, logits + (int64_t)blockIdx.x * TP * C, tile_bytes, &bars[0]);
  }
  __syncthreads();

  int it = 0;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
    const int s = it & 1;
    T* buf = reinterpret_cast<T*>(tile_smem + (size_t)s * stage_stride);
    // queue the next tile into the other stage (its bulk store of two iterations ago has finished reading)
    if (threadIdx.x == 0 && tile + gridDim.x < n_tiles) {
      if (BWD) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      tile_load(tile_smem + (size_t)(s ^ 1) * stage_stride, logits + (tile + gridDim.x) * TP * C, tile_bytes, &bars[s ^ 1]);
    }
    tma::mbar_wait(&bars[s], (uint32_t)((it >> 1) & 1));
    for (int j = 0; j < ppt; ++j) {
    const int px = threadIdx.x / tpc + j * kTileThreads;
    const int rot = rotate ? px % C : 0;
    const int64_t p = tile * TP + px;
    T* row = buf + (size_t)px * C;
    const int lab = load_label<L>(labels, p);
    const bool ign = lab == ignore, ok = (unsigned)lab < (unsigned)C;
    if (!BWD) {
      float m = -FLT_MAX;
      for (int c = part; c < C; c += tpc) {
        int cc = c + rot; cc = cc >= C ? cc - C : cc;
        m = fmaxf(m, to_f32<T>(row[cc]));
      }
      for (int o = 1; o < tpc; o <<= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      const float m2 = m * kLog2e;
      float s0 = 0.f, s1 = 0.f;
      int c = part;
      for (; c + tpc < C; c += 2 * tpc) {
        int ca = c + rot; ca = ca >= C ? ca - C : ca;
        int cb = c + tpc + rot; cb = cb >= C ? cb - C : cb;
        s0 += ex2_approx(fmaf(to_f32<T>(row[ca]), kLog2e, -m2));
        s1 += ex2_approx(fmaf(to_f32<T>(row[cb]), kLog2e, -m2));
      }
      if (c < C) {
        int ca = c + rot; ca = ca >= C ? ca - C : ca;
        s0 += ex2_approx(fmaf(to_f32<T>(row[ca]), kLog2e, -m2));
      }
      float sum = s0 + s1;
      for (int o = 1; o < tpc; o <<= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      if (part == 0) {
        const float lse = m + logf(sum);
        if (!ign && !ok) err |= MDSEG_ERR_LABEL_RANGE;
        const float l = (ok && !ign) ? (lse - to_f32<T>(row[lab])) : 0.f;
        loss_px[p] = l;
        lse_px[p] = lse;
        n_valid += (ok && !ign) ? 1u : 0u;
        if (l > thresh) { ++n_hard; sum_hard += (double)l; }
        ++n_px;
      }
    } else {
      const bool sel = is_selected(sp, loss_px[p]) && ok && !ign;
      const float w = sel ? sp.w : 0.f;
      const float lse2 = lse_px[p] * kLog2e;
      for (int c = part; c < C; c += tpc) {
        int cc = c + rot; cc = cc >= C ? cc - C : cc;
        const float pr = ex2_approx(fmaf(to_f32<T>(row[cc]), kLog2e, -lse2));
        row[cc] = from_f32<T>(w * (pr - ((cc == lab) ? 1.f : 0.f)));
      }
    }
    }  // pixels of this thread
    if (!BWD) {
      __syncthreads();  // every thread has read the stage before it is refilled two iterations later
    } else {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the bulk store
      __syncthreads();
      if (threadIdx.x == 0) {
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dlogits + tile * TP * C),
                     "r"(tma::smem_u32(buf)), "r"(tile_bytes)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    }
  }
  if (BWD) {
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  } else {
    if (err) atomicOr(err_flag, err);
    block_accumulate_stats(st, n_valid, n_hard, sum_hard, n_px);
  }
}

// ---- launchers ----------------------------------------------------------------
int grid_for(int64_t work_items, int per_sm) {
  int64_t blocks = ceil_div64(work_items > 0 ? work_items : 1, 256);
  int64_t cap = (int64_t)sm_count() * per_sm;
  if (blocks > cap) blocks = cap;
  return (int)blocks;
}

template <typename T, typename L>
int launch_fwd(const void* logits, int layout, const void* labels, int N, int C, int H, int W, int ignore,
               float* loss_px, float* lse_px, mdseg_ohem_state* st, int32_t* err_flag, cudaStream_t s) {
  const int64_t HW = (int64_t)H * W;
  if (layout == MDSEG_NHWC) {
    const int64_t P = HW * N;
    // whole tiles through the bulk-copy pipeline, the ragged tail (and shapes whose tile does not fit) warp per pixel
    const int TP = (((uintptr_t)logits & 15) == 0) ? tile_pixels(C, (int)sizeof(T)) : 0;
    const int64_t n_tiles = TP ? P / TP : 0;
    if (n_tiles) {
      const size_t smem = 2 * (((size_t)TP * C * sizeof(T) + 127) & ~(size_t)127);
      auto k = ce_nhwc_tile_kernel<T, L, false>;
      MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      const int grid = (int)(n_tiles < sm_count() ? n_tiles : sm_count());
      k<<<grid, kTileThreads, smem, s>>>((const T*)logits, (const L*)labels, n_tiles, TP, C, ignore, loss_px, lse_px, st,
                                         err_flag, nullptr, 1.f, nullptr);
      MDSEG_LAUNCH_OK();
    }
    const int64_t done = n_tiles * TP;
    if (done < P)
      ce_fwd_nhwc_kernel<T, L><<<grid_for((P - done) * 32, 8), 256, 0, s>>>(
          (const T*)logits + done * C, (const L*)labels + done, P - done, C, ignore, loss_px + done, lse_px + done, st,
          err_flag);
  } else {
    constexpr int PXV = 4;  // four pixels per thread for every dtype (16-byte fp32 / 8-byte 16-bit loads, 8 planes in flight)
    const bool vec = (HW % PXV == 0) && ((((uintptr_t)logits | (uintptr_t)loss_px | (uintptr_t)lse_px) & 15) == 0);
    if (vec)
      ce_fwd_nchw_kernel<T, L, PXV><<<grid_for(HW / PXV * N, 6), 256, 0, s>>>(
          (const T*)logits, (const L*)labels, N, C, HW, ignore, loss_px, lse_px, st, err_flag);
    else
      ce_fwd_nchw_kernel<T, L, 1><<<grid_for(HW * N, 8), 256, 0, s>>>((const T*)logits, (const L*)labels, N, C, HW,
                                                                      ignore, loss_px, lse_px, st, err_flag);
  }
  MDSEG_LAUNCH_OK();
  return 0;
}

template <typename T, typename L>
int launch_bwd(const void* logits, int layout, const void* labels, int N, int C, int H, int W, int ignore,
               const float* loss_px, const float* lse_px, mdseg_ohem_state* st, const float* grad_out,
               float grad_scale, void* dlogits, cudaStream_t s) {
  const int64_t HW = (int64_t)H * W;
  if (layout == MDSEG_NHWC) {
    const int64_t P = HW * N;
    const int TP = ((((uintptr_t)logits | (uintptr_t)dlogits) & 15) == 0) ? tile_pixels(C, (int)sizeof(T)) : 0;
    const int64_t n_tiles = TP ? P / TP : 0;
    if (n_tiles) {
      const size_t smem = 2 * (((size_t)TP * C * sizeof(T) + 127) & ~(size_t)127);
      auto k = ce_nhwc_tile_kernel<T, L, true>;
      MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      const int grid = (int)(n_tiles < sm_count() ? n_tiles : sm_count());
      k<<<grid, kTileThreads, smem, s>>>((const T*)logits, (const L*)labels, n_tiles, TP, C, ignore,
                                         const_cast<float*>(loss_px), const_cast<float*>(lse_px), st, nullptr, grad_out,
                                         grad_scale, (T*)dlogits);
      MDSEG_LAUNCH_OK();
    }
    const int64_t done = n_tiles * TP;
    if (done < P)
      ce_bwd_nhwc_kernel<T, L><<<grid_for((P - done) * 32, 8), 256, 0, s>>>(
          (const T*)logits + done * C, (const L*)labels + done, P - done, C, ignore, loss_px + done, lse_px + done, st,
          grad_out, grad_scale, (T*)dlogits + done * C);
  } else {
    constexpr int PXV = 16 / sizeof(T);
    const bool vec = (HW % PXV == 0) && ((((uintptr_t)logits | (uintptr_t)dlogits) & 15) == 0);
    if (vec)
      ce_bwd_nchw_kernel<T, L, PXV><<<grid_for(HW / PXV * N, 6), 256, 0, s>>>(
          (const T*)logits, (const L*)labels, N, C, HW, ignore, loss_px, lse_px, st, grad_out, grad_scale,
          (T*)dlogits);
    else
      ce_bwd_nchw_kernel<T, L, 1><<<grid_for(HW * N, 8), 256, 0, s>>>((const T*)logits, (const L*)labels, N, C, HW,
                                                                      ignore, loss_px, lse_px, st, grad_out,
                                                                      grad_scale, (T*)dlogits);
  }
  MDSEG_LAUNCH_OK();
  return 0;
}

}  // namespace
}  // namespace mdseg

extern "C" int mdseg_ohem_ce_fwd(const void* logits, int dtype, int layout, const void* labels, int label_dtype,
                                 int N, int C, int H, int W, int ignore, float* loss_px, float* lse_px,
                                 mdseg_ohem_state* state, int32_t* err_flag, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(N >= 0 && C > 0 && H >= 0 && W >= 0, "mdseg_ohem_ce_fwd: bad shape %d %d %d %d", N, C, H, W);
  MDSEG_REQUIRE(layout == MDSEG_NCHW || layout == MDSEG_NHWC, "mdseg_ohem_ce_fwd: bad layout %d", layout);
  if ((int64_t)N * H * W == 0) return 0;
  MDSEG_REQUIRE(logits && labels && loss_px && lse_px && state && err_flag, "mdseg_ohem_ce_fwd: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  return with_float_type(dtype, "mdseg_ohem_ce_fwd", "dtype", [&](auto t) {
    return with_int_type(label_dtype, "mdseg_ohem_ce_fwd", "label dtype", [&](auto l) {
      return launch_fwd<typename decltype(t)::type, typename decltype(l)::type>(
          logits, layout, labels, N, C, H, W, ignore, loss_px, lse_px, state, err_flag, s);
    });
  });
}

extern "C" int mdseg_ohem_ce_bwd(const void* logits, int dtype, int layout, const void* labels, int label_dtype,
                                 int N, int C, int H, int W, int ignore, const float* loss_px, const float* lse_px,
                                 mdseg_ohem_state* state, const float* grad_out, float grad_scale, void* dlogits,
                                 void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(N >= 0 && C > 0 && H >= 0 && W >= 0, "mdseg_ohem_ce_bwd: bad shape");
  MDSEG_REQUIRE(layout == MDSEG_NCHW || layout == MDSEG_NHWC, "mdseg_ohem_ce_bwd: bad layout %d", layout);
  if ((int64_t)N * H * W == 0) return 0;
  MDSEG_REQUIRE(logits && labels && loss_px && lse_px && state && dlogits, "mdseg_ohem_ce_bwd: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  return with_float_type(dtype, "mdseg_ohem_ce_bwd", "dtype", [&](auto t) {
    return with_int_type(label_dtype, "mdseg_ohem_ce_bwd", "label dtype", [&](auto l) {
      return launch_bwd<typename decltype(t)::type, typename decltype(l)::type>(
          logits, layout, labels, N, C, H, W, ignore, loss_px, lse_px, state, grad_out, grad_scale, dlogits, s);
    });
  });
}
