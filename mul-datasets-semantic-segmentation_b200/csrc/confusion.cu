// confusion.cu — confusion-matrix accumulation fused with the label LUT
// (SURVEY §8 rows a12, a13).
//
// Reference work replaced (evaluate.py:89-93,174-181; rectangular variants
// :631-634,1738-1741,1866-1869; tools/evaluate_city.py:72-75):
//   keep = label != 255
//   hist += np.bincount(label[keep]*C + pred[keep], minlength=C*C).view(C,C)
// i.e. 5 D2H copies + a boolean gather + a single-thread bincount + one H2D per
// image.  Here: one pass over (label, pred) in HBM, a privatised shared-memory
// histogram per CTA (replicated per warp when it is small), per-thread
// run-length aggregation of equal consecutive keys (segmentation maps are
// piecewise constant), and one 64-bit global atomic per non-empty bin per CTA.
// The accumulator is int64 (the reference's float32 hist is exact only below
// 2^24 per cell).  Algorithmic bytes per pixel: sizeof(label) + sizeof(pred).
#include "common.cuh"

namespace mdseg {
namespace {

// ---- coalesced warp-chunk loads ---------------------------------------------------------------------------
// A warp walks "chunks" of 32 * kPL consecutive pixels: lane i holds the kPL consecutive pixels starting at
// 32 * kPL * chunk + kPL * i, where kPL * max(sizeof(L), sizeof(P)) = 16 bytes, so every warp-level load is one
// contiguous 512-byte (or narrower) request and each 32-byte sector crosses the L2 -> SM fabric exactly once.
template <typename L, typename P> struct ChunkOf {
  static constexpr int kPL = 16 / (int)(sizeof(L) > sizeof(P) ? sizeof(L) : sizeof(P));
  static constexpr int kUnroll = kPL >= 16 ? 2 : 4;  // chunks in flight per warp
};

// N consecutive elements, kept as raw 32-bit words while the loads are in flight (N * sizeof(T) is 2, 4, 8 or
// 16 bytes) and widened to ints on use; values outside [0, 2^31) become -1.
template <typename T, int N> struct LoadPx {
  static constexpr int kBytes = N * (int)sizeof(T);
  static constexpr int kWords = kBytes < 4 ? 1 : kBytes / 4;
  static_assert(kBytes == 2 || kBytes == 4 || kBytes == 8 || kBytes == 16, "unsupported vector width");
  static __device__ __forceinline__ void load(const T* p, uint32_t (&w)[kWords]) {
    if constexpr (kBytes == 16) {
      const int4 r = ldg_stream_v4(p);
      w[0] = (uint32_t)r.x; w[1] = (uint32_t)r.y; w[2] = (uint32_t)r.z; w[3] = (uint32_t)r.w;
    } else if constexpr (kBytes == 8) {
      const int2 r = ldg_stream_v2(p);
      w[0] = (uint32_t)r.x; w[1] = (uint32_t)r.y;
    } else if constexpr (kBytes == 4) {
      asm volatile("ld.global.nc.L1::no_allocate.b32 %0, [%1];" : "=r"(w[0]) : "l"(p));
    } else {
      unsigned short h;
      asm volatile("ld.global.nc.L1::no_allocate.b16 %0, [%1];" : "=h"(h) : "l"(p));
      w[0] = h;
    }
  }
  static __device__ __forceinline__ int get(const uint32_t (&w)[kWords], int i) {
    if constexpr (sizeof(T) == 1) return (int)((w[i >> 2] >> (8 * (i & 3))) & 0xffu);
    else if constexpr (sizeof(T) == 4) return (int)w[i];
    else return (w[2 * i + 1] == 0u) ? (int)w[2 * i] : -1;
  }
};

// where one CTA's counts go: a privatised shared-memory replica or, for histograms too large for it, HBM
struct HistSink {
  unsigned* sh;               // nullptr -> global
  unsigned long long* glob;
  __device__ __forceinline__ void add(int key, unsigned cnt) const {
    if (sh) atomicAdd(sh + key, cnt);
    else atomicAdd(glob + key, (unsigned long long)cnt);
  }
};

// key of one pixel or -1 (ignored / invalid)
__device__ __forceinline__ int make_key(int l, int p, const uint8_t* s_lut, bool has_lut, int Ca, int Cb, int ignore,
                                        int& err) {
  if (has_lut) {
    if ((unsigned)l < 256u) l = s_lut[l];
    else l = -1;
  }
  if (l == ignore) return -1;
  if ((unsigned)l >= (unsigned)Ca) { err |= MDSEG_ERR_LABEL_RANGE; return -1; }
  if ((unsigned)p >= (unsigned)Cb) { err |= MDSEG_ERR_PRED_RANGE; return -1; }
  return l * Cb + p;
}

// One chunk: run-length aggregation.  Segmentation maps are piecewise constant, so most lanes hold kPL equal
// keys ("uniform" lanes) and most uniform lanes continue their left neighbour's run: the first lane of such a
// run issues ONE atomic for the whole run (its length comes from a ballot of the run boundaries).  Lanes whose
// pixels differ fall back to a private run-length walk.  The shared-memory atomic unit retires about one lane
// every two cycles per SM, which is the floor for maps without any spatial coherence.
template <int N>
__device__ __forceinline__ void warp_chunk_bump(const int (&key)[N], int lane, const HistSink& sink) {
  bool uniform = true;
#pragma unroll
  for (int i = 1; i < N; ++i) uniform &= (key[i] == key[0]);
  const unsigned umask = __ballot_sync(0xffffffffu, uniform);
  const int left = __shfl_up_sync(0xffffffffu, key[0], 1);
  const bool left_uniform = lane > 0 && ((umask >> (lane - 1)) & 1u);
  const bool head = uniform && !(left_uniform && left == key[0]);
  const unsigned boundary = __ballot_sync(0xffffffffu, !uniform || head);
  if (uniform) {
    if (head && key[0] >= 0) {
      const unsigned rest = (lane == 31) ? 0u : (boundary >> (lane + 1));
      const int lanes = rest ? __ffs((int)rest) : (32 - lane);
      sink.add(key[0], (unsigned)(lanes * N));
    }
  } else {
    int prev = key[0];
    unsigned cnt = 1;
#pragma unroll
    for (int i = 1; i < N; ++i) {
      if (key[i] == prev) {
        ++cnt;
      } else {
        if (prev >= 0) sink.add(prev, cnt);
        prev = key[i];
        cnt = 1;
      }
    }
    if (prev >= 0) sink.add(prev, cnt);
  }
}

// All pixels [0, n) of one slice, spread over `n_warps` warps of which this is number `gw`.  `aligned` = both
// pointers are 16-byte aligned (the chunk path); otherwise every pixel is read on its own.
template <typename L, typename P>
__device__ __forceinline__ void accumulate_slice(const L* __restrict__ label, const P* __restrict__ pred, int64_t n,
                                                 bool aligned, int64_t gw, int64_t n_warps, const uint8_t* s_lut,
                                                 bool has_lut, int Ca, int Cb, int ignore, const HistSink& sink,
                                                 int& err) {
  constexpr int kPL = ChunkOf<L, P>::kPL;
  constexpr int kU = ChunkOf<L, P>::kUnroll;
  const int lane = threadIdx.x & 31;
  const int64_t n_chunks = aligned ? n / (32 * kPL) : 0;
  for (int64_t c0 = gw * kU; c0 < n_chunks; c0 += n_warps * kU) {
    uint32_t l[kU][LoadPx<L, kPL>::kWords], p[kU][LoadPx<P, kPL>::kWords];
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      if (c0 + u < n_chunks) {
        const int64_t at = (c0 + u) * (32 * kPL) + lane * kPL;
        LoadPx<L, kPL>::load(label + at, l[u]);
        LoadPx<P, kPL>::load(pred + at, p[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      if (c0 + u < n_chunks) {
        int key[kPL];
#pragma unroll
        for (int i = 0; i < kPL; ++i)
          key[i] = make_key(LoadPx<L, kPL>::get(l[u], i), LoadPx<P, kPL>::get(p[u], i), s_lut, has_lut, Ca, Cb, ignore, err);
        warp_chunk_bump<kPL>(key, lane, sink);
      }
    }
  }
  // ragged tail (and the whole slice when unaligned): one pixel per thread
  for (int64_t i = n_chunks * (32 * kPL) + gw * 32 + lane; i < n; i += n_warps * 32) {
    const int key = make_key(load_label<L>(label, i), load_label<P>(pred, i), s_lut, has_lut, Ca, Cb, ignore, err);
    if (key >= 0) sink.add(key, 1u);
  }
}

constexpr int kConfThreads = 1024;

// Zero `replicas` shared-memory copies of a `bins`-bin histogram / add them into the int64 histogram in HBM.
__device__ __forceinline__ void sh_hist_zero(unsigned* sh, int words) {
  for (int i = threadIdx.x; i < words; i += blockDim.x) sh[i] = 0u;
}
__device__ __forceinline__ void sh_hist_flush(const unsigned* sh, int bins, int replicas, unsigned long long* hist) {
  for (int b = threadIdx.x; b < bins; b += blockDim.x) {
    unsigned long long s = 0;
    for (int r = 0; r < replicas; ++r) s += sh[r * bins + b];
    if (s) atomicAdd(hist + b, s);
  }
}

template <typename L, typename P>
__global__ void __launch_bounds__(kConfThreads)
confusion_kernel(const L* __restrict__ label, const P* __restrict__ pred, const uint8_t* __restrict__ lut,
                 unsigned long long* __restrict__ hist, int Ca, int Cb, int ignore, int64_t n, int* err_flag,
                 int replicas, int aligned) {
  extern __shared__ unsigned sh_hist[];
  __shared__ uint8_t s_lut[256];
  const int bins = Ca * Cb;
  const bool has_lut = lut != nullptr;
  if (has_lut && threadIdx.x < 256) s_lut[threadIdx.x] = lut[threadIdx.x];
  const bool use_smem = replicas > 0;
  if (use_smem) sh_hist_zero(sh_hist, bins * replicas);
  __syncthreads();
  const int warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  HistSink sink{use_smem ? sh_hist + (warp % replicas) * bins : nullptr, hist};
  int err = 0;
  accumulate_slice<L, P>(label, pred, n, aligned != 0, (int64_t)blockIdx.x * warps + warp, (int64_t)gridDim.x * warps,
                         s_lut, has_lut, Ca, Cb, ignore, sink, err);
  if (err) atomicOr(err_flag, err);
  if (use_smem) {
    __syncthreads();
    sh_hist_flush(sh_hist, bins, replicas, hist);
  }
}

// ---- all datasets of a batch in one launch --------------------------------------------------------------
// blockIdx.y = image b; d = dataset_ids[b] selects the LUT (luts + 256*d), the class count C[d] and the
// square histogram hist + offset[d].  Shared-memory privatisation is decided per CTA from C[d].
template <typename L, typename P>
__global__ void __launch_bounds__(kConfThreads)
confusion_images_kernel(const L* __restrict__ label, const P* __restrict__ pred, const uint8_t* __restrict__ luts,
                        const int32_t* __restrict__ dataset_ids, int64_t px_per_image,
                        unsigned long long* __restrict__ hist, const mdseg_hist_table tab, int ignore,
                        int* err_flag, int smem_words) {
  extern __shared__ unsigned sh_hist[];
  __shared__ uint8_t s_lut[256];
  const int b = blockIdx.y;
  const int d = dataset_ids ? dataset_ids[b] : 0;
  if (d < 0 || d >= tab.n_datasets) {
    if (threadIdx.x == 0 && blockIdx.x == 0) atomicOr(err_flag, MDSEG_ERR_DATASET_ID);
    return;
  }
  const int C = tab.C[d];
  const int bins = C * C;
  unsigned long long* h = hist + tab.offset[d];
  const bool has_lut = luts != nullptr;
  if (has_lut && threadIdx.x < 256) s_lut[threadIdx.x] = luts[(int64_t)d * 256 + threadIdx.x];
  const bool use_smem = bins <= smem_words;
  int replicas = 1;
  if (use_smem) {
    replicas = smem_words / bins;
    if (replicas > 8) replicas = 8;
    sh_hist_zero(sh_hist, bins * replicas);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  HistSink sink{use_smem ? sh_hist + (warp % replicas) * bins : nullptr, h};
  int err = 0;
  // the host guarantees 16-byte aligned image slices
  accumulate_slice<L, P>(label + (int64_t)b * px_per_image, pred + (int64_t)b * px_per_image, px_per_image, true,
                         (int64_t)blockIdx.x * warps + warp, (int64_t)gridDim.x * warps, s_lut, has_lut, C, C, ignore,
                         sink, err);
  if (err) atomicOr(err_flag, err);
  if (use_smem) {
    __syncthreads();
    sh_hist_flush(sh_hist, bins, replicas, h);
  }
}

// iou / mIoU of every dataset: one CTA per dataset.  Row / column sums are coalesced (a warp walks a row,
// lanes walk columns); the nanmean is a fixed-shape shuffle tree in double, so it is run-to-run deterministic.
__global__ void __launch_bounds__(256) miou_images_kernel(const long long* __restrict__ hist, const mdseg_hist_table tab,
                                                          float* __restrict__ iou, int iou_stride,
                                                          float* __restrict__ miou) {
  extern __shared__ long long s_sum[];  // [2][C]: row sums, column sums
  const int d = blockIdx.x;
  const int C = tab.C[d];
  const long long* h = hist + tab.offset[d];
  float* io = iou + (int64_t)d * iou_stride;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  long long* rows = s_sum;
  long long* cols = s_sum + C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) cols[c] = 0;
  __syncthreads();
  for (int r = warp; r < C; r += n_warps) {  // warp r-th row: coalesced; column partials kept per lane
    long long acc = 0;
    for (int j = lane; j < C; j += 32) {
      const long long v = h[(int64_t)r * C + j];
      acc += v;
      if (v) atomicAdd(reinterpret_cast<unsigned long long*>(&cols[j]), (unsigned long long)v);  // integer: exact
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) rows[r] = acc;
  }
  __syncthreads();
  double part = 0.0;
  int cnt = 0;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const long long dg = h[(int64_t)c * C + c];
    // evaluate.py:96: diag / (sum0 + sum1 - diag); 0/0 -> NaN (class absent)
    const float v = (float)((double)dg / (double)(cols[c] + rows[c] - dg));
    io[c] = v;
    if (v == v) { part += (double)v; ++cnt; }
  }
  __shared__ double s_part[8];
  __shared__ int s_cnt[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    part += __shfl_xor_sync(0xffffffffu, part, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if (lane == 0) { s_part[warp] = part; s_cnt[warp] = cnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double sum = 0.0;
    int n = 0;
    for (int w = 0; w < n_warps; ++w) { sum += s_part[w]; n += s_cnt[w]; }
    miou[d] = n ? (float)(sum / n) : __int_as_float(0x7fc00000);
  }
}

// Grid shape shared by both launchers: one 1024-thread CTA per SM (32 warps keep ~128 KB of loads in flight and
// halve the number of per-CTA histogram flushes compared with two smaller CTAs), the images' CTA count rounded
// DOWN so that the whole grid is resident at once (a second, nearly empty wave would double the run time).
template <typename L, typename P>
int launch_images(const void* label, const void* pred, const uint8_t* luts, const int32_t* ids, int n_images,
                  int64_t ppi, int64_t* hist, const mdseg_hist_table& tab, int ignore, int32_t* err_flag,
                  cudaStream_t st) {
  int cmax = 0;
  for (int i = 0; i < tab.n_datasets; ++i) cmax = tab.C[i] > cmax ? tab.C[i] : cmax;
  // privatised histogram: up to 32 KB of replicas for small C, one replica up to 200 KB, global atomics beyond
  size_t smem = (size_t)cmax * cmax * 4;
  if (smem < 32 * 1024) smem = 32 * 1024;
  if (smem > 200 * 1024) smem = 32 * 1024;
  auto k = confusion_images_kernel<L, P>;
  if (smem > 48 * 1024) MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = smem <= 100 * 1024 ? 2 : 1;  // 2 x 1024 threads is the SM's thread limit
  constexpr int kPxPerCtaIter = (kConfThreads / 32) * 32 * ChunkOf<L, P>::kPL * ChunkOf<L, P>::kUnroll;
  int64_t blocks = ceil_div64(ppi, kPxPerCtaIter);
  const int64_t cap = ((int64_t)sm_count() * per_sm) / n_images;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  k<<<dim3((unsigned)blocks, (unsigned)n_images), kConfThreads, smem, st>>>(
      (const L*)label, (const P*)pred, luts, ids, ppi, reinterpret_cast<unsigned long long*>(hist), tab, ignore,
      err_flag, (int)(smem / 4));
  MDSEG_LAUNCH_OK();
  return 0;
}

template <typename L, typename P>
int launch(const void* label, const void* pred, const uint8_t* lut, int64_t* hist, int Ca, int Cb, int ignore,
           int64_t n, int32_t* err_flag, cudaStream_t st) {
  const int64_t bins = (int64_t)Ca * Cb;
  const bool aligned = (((uintptr_t)label | (uintptr_t)pred) & 15) == 0;
  const size_t kMaxSmem = 200 * 1024;
  int replicas = 0;  // 0: histogram too large for shared memory, global atomics
  size_t smem = 0;
  int per_sm = 2;
  if ((size_t)bins * 4 <= kMaxSmem) {
    replicas = (int)((32 * 1024) / (bins * 4));
    if (replicas > 8) replicas = 8;
    if (replicas < 1) replicas = 1;
    smem = (size_t)bins * 4 * replicas;
    if (smem > 100 * 1024) per_sm = 1;
  }
  constexpr int kPxPerCtaIter = (kConfThreads / 32) * 32 * ChunkOf<L, P>::kPL * ChunkOf<L, P>::kUnroll;
  int64_t blocks = ceil_div64(n, kPxPerCtaIter);
  const int64_t cap = (int64_t)sm_count() * per_sm;
  if (blocks > cap) blocks = cap;
  auto k = confusion_kernel<L, P>;
  if (smem > 48 * 1024) MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<(unsigned)blocks, kConfThreads, smem, st>>>((const L*)label, (const P*)pred, lut,
                                                  reinterpret_cast<unsigned long long*>(hist), Ca, Cb, ignore, n,
                                                  err_flag, replicas, aligned ? 1 : 0);
  MDSEG_LAUNCH_OK();
  return 0;
}

// iou / mIoU on the device: one CTA; the final nanmean is a sequential double
// sum by one thread so the result is run-to-run deterministic.
__global__ void miou_kernel(const long long* __restrict__ hist, int C, float* __restrict__ iou,
                            float* __restrict__ miou) {
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    long long row = 0, col = 0;
    for (int j = 0; j < C; ++j) { row += hist[(int64_t)c * C + j]; col += hist[(int64_t)j * C + c]; }
    long long d = hist[(int64_t)c * C + c];
    // evaluate.py:96: diag / (sum0 + sum1 - diag); 0/0 -> NaN (class absent)
    iou[c] = (float)((double)d / (double)(col + row - d));
  }
  __syncthreads();
  if (threadIdx.x == 0 && miou) {
    double s = 0.0;
    int cnt = 0;
    for (int c = 0; c < C; ++c) {
      float v = iou[c];
      if (v == v) { s += (double)v; ++cnt; }
    }
    *miou = cnt ? (float)(s / cnt) : __int_as_float(0x7fc00000);
  }
}

}  // namespace
}  // namespace mdseg

extern "C" int mdseg_confusion(const void* label, int label_dtype, const void* pred, int pred_dtype,
                               const uint8_t* lut256, int64_t* hist, int Ca, int Cb, int ignore, int64_t n,
                               int32_t* err_flag, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(Ca > 0 && Cb > 0 && (int64_t)Ca * Cb < (1LL << 31), "mdseg_confusion: bad Ca/Cb %d %d", Ca, Cb);
  MDSEG_REQUIRE(n >= 0, "mdseg_confusion: n < 0");
  if (n == 0) return 0;
  MDSEG_REQUIRE(label && pred && hist && err_flag, "mdseg_confusion: null pointer (err_flag is required)");
  cudaStream_t st = (cudaStream_t)stream;
  return with_int_type(label_dtype, "mdseg_confusion", "label_dtype", [&](auto l) {
    return with_int_type(pred_dtype, "mdseg_confusion", "pred_dtype", [&](auto p) {
      return launch<typename decltype(l)::type, typename decltype(p)::type>(label, pred, lut256, hist, Ca, Cb, ignore,
                                                                            n, err_flag, st);
    });
  });
}

extern "C" int mdseg_miou(const int64_t* hist, int C, float* iou, float* miou, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(hist && iou && C > 0, "mdseg_miou: bad arguments (iou is required)");
  miou_kernel<<<1, 256, 0, (cudaStream_t)stream>>>((const long long*)hist, C, iou, miou);
  MDSEG_LAUNCH_OK();
  return 0;
}

extern "C" int mdseg_confusion_images(const void* label, int label_dtype, const void* pred, int pred_dtype,
                                      const uint8_t* luts, const int32_t* dataset_ids, int n_images,
                                      int64_t px_per_image, int64_t* hist, const mdseg_hist_table* tab, int ignore,
                                      int32_t* err_flag, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(tab && tab->n_datasets > 0 && tab->n_datasets <= MDSEG_MAX_DATASETS, "mdseg_confusion_images: bad table");
  for (int i = 0; i < tab->n_datasets; ++i)
    MDSEG_REQUIRE(tab->C[i] > 0 && tab->C[i] < 32768 && tab->offset[i] >= 0, "mdseg_confusion_images: bad table entry %d", i);
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && px_per_image >= 0, "mdseg_confusion_images: bad shape");
  if (n_images == 0 || px_per_image == 0) return 0;
  MDSEG_REQUIRE(label && pred && hist && err_flag, "mdseg_confusion_images: null pointer (err_flag is required)");
  MDSEG_REQUIRE(px_per_image % 16 == 0 && (((uintptr_t)label | (uintptr_t)pred) & 15) == 0,
                "mdseg_confusion_images: images must be 16-element multiples and 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  return with_int_type(label_dtype, "mdseg_confusion_images", "label_dtype", [&](auto l) {
    return with_int_type(pred_dtype, "mdseg_confusion_images", "pred_dtype", [&](auto p) {
      return launch_images<typename decltype(l)::type, typename decltype(p)::type>(
          label, pred, luts, dataset_ids, n_images, px_per_image, hist, *tab, ignore, err_flag, st);
    });
  });
}

extern "C" int mdseg_miou_images(const int64_t* hist, const mdseg_hist_table* tab, float* iou, int iou_stride,
                                 float* miou, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(hist && tab && iou && miou && tab->n_datasets > 0 && tab->n_datasets <= MDSEG_MAX_DATASETS,
                "mdseg_miou_images: bad arguments");
  for (int i = 0; i < tab->n_datasets; ++i)
    MDSEG_REQUIRE(tab->C[i] > 0 && tab->C[i] <= iou_stride, "mdseg_miou_images: iou_stride %d < C[%d]", iou_stride, i);
  int cmax = 0;
  for (int i = 0; i < tab->n_datasets; ++i) cmax = tab->C[i] > cmax ? tab->C[i] : cmax;
  MDSEG_REQUIRE((size_t)cmax * 16 <= 48 * 1024, "mdseg_miou_images: more than 3072 classes");
  miou_images_kernel<<<tab->n_datasets, 256, (size_t)cmax * 16, (cudaStream_t)stream>>>((const long long*)hist, *tab,
                                                                                       iou, iou_stride, miou);
  MDSEG_LAUNCH_OK();
  return 0;
}
