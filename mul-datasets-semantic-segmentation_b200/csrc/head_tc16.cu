// head_tc16.cu — the prototype head for 16-bit features (AMP: fp16 / bf16) as a TMA-fed, warp-specialised tcgen05 GEMM
// (SURVEY §8 row f2; VERDICT r1 items 6 / 7).
//
// Reference work replaced (lib/models/semseg.py:325-333,342-343; lib/loss/loss_cross_datasets.py:950,961,971 under
// amp.autocast):   logits = torch.einsum('bchw, nc -> bnhw', feats, unify_prototype)
//
// GEMM per CTA:  D[M = 128 pixels, N = NT prototypes (<= 256)] = sum_k A[m, k] * B[n, k],  K = feature channels.
//   * A = feats is NCHW: for one channel the pixels are contiguous, i.e. A is MN-MAJOR.  It is never transposed or
//     touched by a thread: TMA boxes [64 channels][64 pixels] land in shared memory in the canonical MN-major
//     128-byte-swizzle layout (two boxes = 128 pixels) and the UMMA reads them with a_major = MN.
//   * B = prototypes [N, K] (K-major), converted once to the feature dtype and zero-padded to whole N tiles by the
//     host side; TMA boxes [NT rows][64 k], 128-byte swizzle.
//   * roles: warp 0 lane 0 = TMA producer, warp 1 lane 0 = MMA issuer (tcgen05.mma kind::f16, fp32 accumulator in
//     TMEM, tcgen05.commit releases the stage), warps 2-5 = epilogue (tcgen05.ld 32x32b: a TMEM lane is a pixel, so a
//     warp stores 32 consecutive pixels of one prototype plane per instruction).
//   * two CTAs per SM (two 40 KB stages and 256 TMEM columns each): one CTA's epilogue overlaps the other's main loop.
// The N tiles of one pixel tile are neighbouring CTAs (blockIdx.x), so the second read of A comes from L2.
//
// Pixel-major (channels_last, NHWC) variants, chosen at compile time so that the MMA issue loop never branches on them:
//   * kAK: A = x [n_images, hw, K] — the channel is contiguous, i.e. A is K-MAJOR, exactly like B: one TMA box
//     [128 pixels][64 channels] (16 KB, the same kABytes) per stage, 128-byte swizzle, a_major = K.
//   * kOutPM: the output is [n_images, hw, out_cstride] — a TMEM lane is a pixel and its columns are channels, so an
//     epilogue thread writes 16 consecutive channels of its pixel (32 B in 16 bit, 64 B in fp32) as 16-byte stores.
//   * head_tc16_dw_kernel<true> reads feats [n_images, hw, K] as its B operand (N = channels, K = pixels): MN-MAJOR,
//     staged as ceil(NT / 64) TMA boxes [64 pixels][64 channels], the layout the forward uses for its MN-major A.
// The tensor cores see the same 16-bit products in the same K order as on the planar layout, so every output of the
// pixel-major variants is bit-identical to the planar one on x.contiguous().  The entry points take the layout of x
// (MDSEG_NCHW / MDSEG_NHWC) as an argument and pick the variant from it.
#include "tma_util.cuh"

namespace mdseg {
namespace {

using namespace tma;

constexpr int kM = 128;           // pixels per tile (UMMA M)
constexpr int kKB = 64;           // channels per stage: 64 x 2 B = one 128-byte swizzle row of B
constexpr int kNStages = 2;
constexpr int kThreads = 192;     // producer warp, MMA warp, four epilogue warps
constexpr int kABytes = kKB * kM * 2;  // 16 KB: [2 pixel atoms][64 channel rows][128 B]

struct HeadArgs {
  void* out;          // [n_images, out_cstride, hw] (kOutPM: [n_images, hw, out_cstride]) fp32 or the feature dtype
  long long hw;
  const int32_t* dataset_ids;  // NULL: every image uses B operand 0
  int Nd[MDSEG_MAX_DATASETS], NTd[MDSEG_MAX_DATASETS];  // output rows / N tile width per B operand
  int n_datasets, out_cstride, n_kb, fmt;
  int zero_N, zero_NT;  // zero_N > 0: images of no dataset get zeros in their zero_N output rows (tiles of zero_NT)
};

// 16 channels of one pixel, pixel-major output: whole 16-byte stores (o is 32-byte aligned)
template <typename TO>
__device__ __forceinline__ void store16_pm(TO* o, const uint32_t* r) {
  uint4* v = reinterpret_cast<uint4*>(o);
  if constexpr (sizeof(TO) == 4) {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = make_uint4(r[4 * i], r[4 * i + 1], r[4 * i + 2], r[4 * i + 3]);
  } else {
    uint32_t w[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const TO lo = from_f32<TO>(__uint_as_float(r[2 * i])), hi = from_f32<TO>(__uint_as_float(r[2 * i + 1]));
      w[i] = (uint32_t)(*reinterpret_cast<const unsigned short*>(&lo)) |
             ((uint32_t)(*reinterpret_cast<const unsigned short*>(&hi)) << 16);
    }
    v[0] = make_uint4(w[0], w[1], w[2], w[3]);
    v[1] = make_uint4(w[4], w[5], w[6], w[7]);
  }
}

template <typename TO, bool kAK, bool kOutPM>
__global__ void __launch_bounds__(kThreads, 2) head_tc16_kernel(const __grid_constant__ CUtensorMap mapA,
                                                                const __grid_constant__ Maps mapsB,
                                                                const __grid_constant__ HeadArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ __align__(8) uint64_t full[kNStages], empty[kNStages], acc_full;
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nz = blockIdx.x, b = blockIdx.z;
  const long long p0 = (long long)blockIdx.y * kM;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  if (d < 0 || d >= a.n_datasets) {                 // uniform per CTA: an image of no dataset
    if (a.zero_N > 0) {                             // gradient route: its rows are zero (else the caller zero-fills)
      const int n0 = nz * a.zero_NT;
      if constexpr (kOutPM) {  // rows [p0, p0 + 128) x channels [n0, n0 + zero_NT): consecutive threads, consecutive channels
        TO* ob = (TO*)a.out + (long long)b * a.hw * a.out_cstride + n0;
        for (int i = threadIdx.x; i < a.zero_NT * kM; i += kThreads) {
          const int r = i / a.zero_NT, c = i - r * a.zero_NT;
          const long long p = p0 + r;
          if (n0 + c < a.zero_N && p < a.hw) ob[p * a.out_cstride + c] = from_f32<TO>(0.f);
        }
      } else {
        TO* ob = (TO*)a.out + ((long long)b * a.out_cstride + n0) * a.hw;
        for (int i = threadIdx.x; i < a.zero_NT * kM; i += kThreads) {
          const int c = i / kM;
          const long long p = p0 + (i - c * kM);
          if (n0 + c < a.zero_N && p < a.hw) ob[(long long)c * a.hw + p] = from_f32<TO>(0.f);
        }
      }
    }
    return;
  }
  const int NT = a.NTd[d], Nout = a.Nd[d];
  if (NT == 0 || nz * NT >= Nout) return;
  const CUtensorMap& mapB = mapsB.m[d];  // the B operand: prototypes, or the dense graph of dataset d
  const uint32_t b_bytes = (uint32_t)NT * 128u;
  const uint32_t stage_bytes = kABytes + b_bytes;
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < NT) tmem_cols <<= 1;

  if (threadIdx.x == 0) {
    prefetch_map(&mapA);
    prefetch_map(&mapB);
    for (int s = 0; s < kNStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(&acc_full, 1);
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(&tmem_base_s, tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = tmem_base_s;

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < a.n_kb; ++kb) {
        const int s = kb % kNStages;
        if (kb >= kNStages) mbar_wait(&empty[s], (uint32_t)((kb / kNStages - 1) & 1));
        unsigned char* st = smem + (size_t)s * stage_bytes;
        mbar_expect_tx(&full[s], stage_bytes);
        if constexpr (kAK) {
          load_3d(st, &mapA, &full[s], kb * kKB, (int)p0, b);                   // [128 pixels][64 channels]
        } else {
          load_3d(st, &mapA, &full[s], (int)p0, kb * kKB, b);                   // pixels p0 .. p0+63
          load_3d(st + kKB * 128, &mapA, &full[s], (int)p0 + 64, kb * kKB, b);  // pixels p0+64 .. p0+127
        }
        load_2d(st + kABytes, &mapB, &full[s], kb * kKB, nz * NT);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // instruction descriptor: fp32 accumulate, A MN-major (bit 15; clear for kAK), B K-major, N = NT, M = 128
      const uint32_t idesc = (1u << 4) | ((uint32_t)a.fmt << 7) | ((uint32_t)a.fmt << 10) | (kAK ? 0u : (1u << 15)) |
                             ((uint32_t)(NT >> 3) << 17) | ((uint32_t)(kM >> 4) << 24);
      for (int kb = 0; kb < a.n_kb; ++kb) {
        const int s = kb % kNStages;
        mbar_wait(&full[s], (uint32_t)((kb / kNStages) & 1));
        tc_fence_after();
        const uint32_t aA = smem_u32(smem + (size_t)s * stage_bytes), aB = aA + kABytes;
#pragma unroll
        for (int ks = 0; ks < kKB / 16; ++ks) {
          // A (MN-major): 16 channels = two 8-row atoms of 1024 B; the second 64-pixel atom kKB * 128 B further on.
          // A (kAK, K-major): like B — 16 channels = 32 bytes inside the swizzle row; 8-pixel groups 1024 B apart
          const uint64_t ad = kAK ? umma_desc(aA + ks * 32, 16, 1024, kSwizzle128B)
                                  : umma_desc(aA + ks * 2048, kKB * 128, 1024, kSwizzle128B);
          // B (K-major): 16 k = 32 bytes inside the 128-byte swizzle row; 8-row groups 1024 B apart
          const uint64_t bd = umma_desc(aB + ks * 32, 16, 1024, kSwizzle128B);
          umma_f16(tmem_d, ad, bd, idesc, (kb > 0 || ks > 0) ? 1u : 0u);
        }
        tc_commit(&empty[s]);
        if (kb == a.n_kb - 1) tc_commit(&acc_full);
      }
    }
  } else {
    // epilogue: warp w may touch TMEM lanes 32 (w % 4) .. + 31
    const int q = warp & 3;
    const long long p = p0 + q * 32 + lane;
    mbar_wait(&acc_full, 0);
    tc_fence_after();
    const int n0 = nz * NT;
    TO* ob = (TO*)a.out + ((long long)b * a.out_cstride + n0) * a.hw;  // planar output
    // 16 accumulator columns per TMEM load, two register sets: the load of the next 16 columns is in flight while the
    // current ones are stored (a load + wait + 16 stores in lockstep left the four epilogue warps waiting on TMEM
    // latency for about half of the epilogue).  The wait names the registers it releases, so no use can move above it.
    int n_eff = Nout - n0;
    n_eff = n_eff > NT ? NT : (n_eff + 15) & ~15;
    const uint32_t taddr = tmem_d + ((uint32_t)(q * 32) << 16);
    uint32_t ra[16], rb[16];
#define MDSEG_H16_ST(R, C0)                                                                                            \
  if constexpr (kOutPM) {                                                                                              \
    if (p < a.hw) {                                                                                                    \
      TO* o = (TO*)a.out + ((long long)b * a.hw + p) * a.out_cstride + n0 + (C0);                                      \
      if (n0 + (C0) + 16 <= Nout) {                                                                                    \
        store16_pm<TO>(o, R);                                                                                          \
      } else {                                                                                                         \
        _Pragma("unroll") for (int i = 0; i < 16; ++i)                                                                 \
          if (n0 + (C0) + i < Nout) o[i] = from_f32<TO>(__uint_as_float(R[i]));                                        \
      }                                                                                                                \
    }                                                                                                                  \
  } else if (p < a.hw) {                                                                                               \
    TO* o = ob + (long long)(C0) * a.hw + p;                                                                           \
    if (n0 + (C0) + 16 <= Nout) { /* whole group inside the output: no per-column test */                              \
      _Pragma("unroll") for (int i = 0; i < 16; ++i) { *o = from_f32<TO>(__uint_as_float(R[i])); o += a.hw; }          \
    } else {                                                                                                           \
      _Pragma("unroll") for (int i = 0; i < 16; ++i) {                                                                 \
        if (n0 + (C0) + i < Nout) *o = from_f32<TO>(__uint_as_float(R[i]));                                            \
        o += a.hw;                                                                                                     \
      }                                                                                                                \
    }                                                                                                                  \
  }
    if (n_eff > 0) tmem_ld16(taddr, ra);
    for (int c0 = 0; c0 < n_eff; c0 += 32) {
      tmem_wait_ld(ra);
      const bool has_b = c0 + 16 < n_eff;
      if (has_b) tmem_ld16(taddr + (uint32_t)(c0 + 16), rb);
      MDSEG_H16_ST(ra, c0);
      if (has_b) {
        tmem_wait_ld(rb);
        if (c0 + 32 < n_eff) tmem_ld16(taddr + (uint32_t)(c0 + 32), ra);
        MDSEG_H16_ST(rb, c0 + 16);
      }
    }
#undef MDSEG_H16_ST
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_d, tmem_cols);
}

// ---- d prototype: dW[n, k] = sum over images and pixels of dy[b, n, p] * feats[b, k, p] -------------------------
// Both operands have the contraction index (the pixel) contiguous: two K-major TMA operands, no transposition.
// A CTA takes one 128-row tile of prototypes, one NT-column tile of feature channels and one slab of the pixels of
// one image; its fp32 partial goes to a workspace slot and a second kernel adds the slots in a fixed order
// (deterministic).  The tile CTAs of one slab are neighbours in the grid, so operand re-reads hit L2.
// kBMN: feats is pixel-major [n_images, hw, K], so B is MN-major (the channel is contiguous): ceil(NT / 64) TMA boxes
// [64 pixels][64 channels] per stage, b_major = MN.  Columns of the last box past NT are loaded and never read.
struct DwArgs {
  float* part;        // [n_slabs_total][m_tiles][n_tiles][128][NT]
  long long hw, slab; // pixels per image, pixels per slab (multiple of 64)
  int slabs_per_image, m_tiles, n_tiles, NT, fmt;
};

template <bool kBMN>
__global__ void __launch_bounds__(kThreads, 2) head_tc16_dw_kernel(const __grid_constant__ CUtensorMap mapA,
                                                                   const __grid_constant__ CUtensorMap mapB,
                                                                   const __grid_constant__ DwArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ __align__(8) uint64_t full[kNStages], empty[kNStages], acc_full;
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x, mt = tile / a.n_tiles, nt = tile % a.n_tiles;
  const int slab_id = blockIdx.y, b = slab_id / a.slabs_per_image, sl = slab_id % a.slabs_per_image;
  const long long p_beg = (long long)sl * a.slab;
  const long long p_end = (p_beg + a.slab < a.hw) ? p_beg + a.slab : a.hw;
  const int n_kb = (int)((p_end - p_beg + 63) / 64);
  const int NT = a.NT;
  constexpr uint32_t a_bytes = 128 * 128;  // [128 prototype rows][64 px x 2 B]
  const int n_boxes = (NT + 63) / 64;  // kBMN: 64-channel boxes of B per stage
  const uint32_t stage_bytes = a_bytes + (kBMN ? (uint32_t)n_boxes * 8192u : (uint32_t)NT * 128u);
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < NT) tmem_cols <<= 1;

  if (threadIdx.x == 0) {
    prefetch_map(&mapA);
    prefetch_map(&mapB);
    for (int s = 0; s < kNStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(&acc_full, 1);
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(&tmem_base_s, tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = tmem_base_s;

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < n_kb; ++kb) {
        const int s = kb % kNStages;
        if (kb >= kNStages) mbar_wait(&empty[s], (uint32_t)((kb / kNStages - 1) & 1));
        unsigned char* st = smem + (size_t)s * stage_bytes;
        mbar_expect_tx(&full[s], stage_bytes);
        // pixels beyond the slab but inside the image would be counted twice: slabs are whole 64-pixel chunks, and
        // pixels beyond the image are zero-filled by TMA
        load_3d(st, &mapA, &full[s], (int)(p_beg + (long long)kb * 64), mt * 128, b);
        if constexpr (kBMN) {
          for (int j = 0; j < n_boxes; ++j)
            load_3d(st + a_bytes + j * 8192, &mapB, &full[s], nt * NT + 64 * j, (int)(p_beg + (long long)kb * 64), b);
        } else {
          load_3d(st + a_bytes, &mapB, &full[s], (int)(p_beg + (long long)kb * 64), nt * NT, b);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // fp32 accumulate, A K-major, B K-major (kBMN: MN-major, bit 16), N = NT, M = 128
      const uint32_t idesc = (1u << 4) | ((uint32_t)a.fmt << 7) | ((uint32_t)a.fmt << 10) | (kBMN ? (1u << 16) : 0u) |
                             ((uint32_t)(NT >> 3) << 17) | ((uint32_t)(kM >> 4) << 24);
      for (int kb = 0; kb < n_kb; ++kb) {
        const int s = kb % kNStages;
        mbar_wait(&full[s], (uint32_t)((kb / kNStages) & 1));
        tc_fence_after();
        const uint32_t aA = smem_u32(smem + (size_t)s * stage_bytes), aB = aA + a_bytes;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks)
          // kBMN: 16 pixels = two 8-row atoms of 1024 B; the next 64-channel atom one 8 KB box further on
          umma_f16(tmem_d, umma_desc(aA + ks * 32, 16, 1024, kSwizzle128B),
                   kBMN ? umma_desc(aB + ks * 2048, 64 * 128, 1024, kSwizzle128B)
                        : umma_desc(aB + ks * 32, 16, 1024, kSwizzle128B),
                   idesc, (kb > 0 || ks > 0) ? 1u : 0u);
        tc_commit(&empty[s]);
        if (kb == n_kb - 1) tc_commit(&acc_full);
      }
    }
  } else {
    const int q = warp & 3;
    const int row = q * 32 + lane;
    mbar_wait(&acc_full, 0);
    tc_fence_after();
    float* slot = a.part + ((((long long)slab_id * a.m_tiles + mt) * a.n_tiles + nt) * 128 + row) * NT;
    for (int c0 = 0; c0 < NT; c0 += 16) {
      uint32_t r[16];
      tmem_ld16(tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, r);
      tmem_wait_ld();
      uint4* o = reinterpret_cast<uint4*>(slot + c0);
#pragma unroll
      for (int i = 0; i < 4; ++i) o[i] = make_uint4(r[4 * i], r[4 * i + 1], r[4 * i + 2], r[4 * i + 3]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_d, tmem_cols);
}

// dataset_ids == NULL: one sum over every slab -> dW [N, K].  Otherwise blockIdx.y is a dataset and only the slabs of
// its images are added -> dW [n_datasets, N, K] (d bi_graph of the dense projection, one matrix per dataset).
__global__ void __launch_bounds__(256) head_tc16_dw_reduce_kernel(const DwArgs a, int n_slabs_total, int N, int K,
                                                                  const int32_t* __restrict__ dataset_ids,
                                                                  float* __restrict__ dW) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * K) return;
  const int n = idx / K, k = idx - n * K;
  const int mt = n / 128, r = n - mt * 128, nt = k / a.NT, c = k - nt * a.NT;
  const int d = (int)blockIdx.y;
  float sum = 0.f;
  for (int s = 0; s < n_slabs_total; ++s) {
    if (dataset_ids != nullptr && dataset_ids[s / a.slabs_per_image] != d) continue;
    sum += a.part[((((long long)s * a.m_tiles + mt) * a.n_tiles + nt) * 128 + r) * a.NT + c];
  }
  dW[(long long)d * N * K + idx] = sum;
}

// the TMA encoder, with the primary context current on the calling thread; NULL (error set) if either is missing
tma::EncodeTiledFn tensor_map_encoder() {
  const tma::EncodeTiledFn enc = tma::encode_fn();
  if (enc == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available in this driver");
    return nullptr;
  }
  return tma::bind_primary_context() ? nullptr : enc;
}

}  // namespace
}  // namespace mdseg

// N tile width for N prototypes: equal tiles of at most 256 rows, multiple of 16
extern "C" int mdseg_head_tc16_tile(int N) {
  if (N <= 0) return 0;
  const int n_tiles = (((N + 15) & ~15) + 255) / 256;
  return (((N + n_tiles - 1) / n_tiles) + 15) & ~15;
}

namespace mdseg {
namespace {
template <typename TO, bool kAK, bool kOutPM>
int launch_head16_kernel(const CUtensorMap& mapA, const Maps& mapsB, const HeadArgs& a, dim3 grid, size_t smem,
                         cudaStream_t s) {
  auto k = head_tc16_kernel<TO, kAK, kOutPM>;
  MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<grid, kThreads, smem, s>>>(mapA, mapsB, a);
  return 0;
}

// A = x [n_images, K, hw] (16-bit, MN-major by TMA) or, a_pm, [n_images, hw, K] (K-major); B operand d = bt[d]:
// [n_tiles(d) * NT(d), ldb] in the same dtype.  out: [n_images, out_cstride, hw] or, out_pm, [n_images, hw, out_cstride]
int launch_head16(const void* x, int dtype, int n_images, int K, int64_t hw, const void* const* bt, int ldb, const int* Nd,
                  int n_b, const int32_t* dataset_ids, void* out, int out_cstride, int out_dtype, cudaStream_t s,
                  const char* who, int zero_N = 0, bool a_pm = false, bool out_pm = false) {
  MDSEG_REQUIRE(dtype == MDSEG_BF16 || dtype == MDSEG_F16, "%s: inputs must be bf16 or fp16", who);
  MDSEG_REQUIRE(out_dtype == MDSEG_F32 || out_dtype == dtype, "%s: output is fp32 or the input dtype", who);
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && K > 0 && hw > 0 && n_b > 0 && n_b <= MDSEG_MAX_DATASETS, "%s: bad shape", who);
  MDSEG_REQUIRE(ldb >= K && ldb % 8 == 0 && hw % 8 == 0,
                "%s: ldb and h * w must be multiples of 8 (16-byte TMA strides), ldb >= K", who);
  MDSEG_REQUIRE(!a_pm || K % 8 == 0, "%s: the channel count of pixel-major x must be a multiple of 8 (16-byte TMA pixel "
                "stride)", who);
  MDSEG_REQUIRE(!out_pm || out_cstride % 8 == 0, "%s: the channel count of a pixel-major output must be a multiple of 8",
                who);
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(x && out && bt && Nd, "%s: null pointer", who);
  MDSEG_REQUIRE(((uintptr_t)x & 15) == 0, "%s: operands must be 16-byte aligned", who);
  MDSEG_REQUIRE(!out_pm || ((uintptr_t)out & 15) == 0, "%s: a pixel-major output must be 16-byte aligned", who);
  const tma::EncodeTiledFn enc = tensor_map_encoder();
  if (enc == nullptr) return 1;
  const CUtensorMapDataType dt = dtype == MDSEG_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUtensorMap mapA;
  {
    cuuint64_t dims[3] = {(cuuint64_t)hw, (cuuint64_t)K, (cuuint64_t)n_images};
    cuuint64_t strides[2] = {(cuuint64_t)hw * 2, (cuuint64_t)K * hw * 2};
    cuuint32_t box[3] = {64, (cuuint32_t)kKB, 1};
    if (a_pm) {  // [n_images, hw, K]: one box of [128 pixels][64 channels]
      dims[0] = (cuuint64_t)K; dims[1] = (cuuint64_t)hw;
      strides[0] = (cuuint64_t)K * 2;
      box[0] = (cuuint32_t)kKB; box[1] = (cuuint32_t)kM;
    }
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(&mapA, dt, 3, const_cast<void*>(x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MDSEG_REQUIRE(r == CUDA_SUCCESS, "%s: cuTensorMapEncodeTiled failed for the A operand (CUresult %d)", who, (int)r);
  }
  Maps mapsB;
  HeadArgs a;
  a.out = out; a.hw = hw; a.dataset_ids = dataset_ids; a.n_datasets = n_b; a.out_cstride = out_cstride;
  a.n_kb = (K + kKB - 1) / kKB;
  a.fmt = dtype == MDSEG_F16 ? 0 : 1;
  a.zero_N = zero_N; a.zero_NT = mdseg_head_tc16_tile(zero_N);
  int tiles_max = 0, nt_max = 0;
  if (zero_N > 0) { tiles_max = (zero_N + a.zero_NT - 1) / a.zero_NT; nt_max = a.zero_NT; }
  for (int d = 0; d < MDSEG_MAX_DATASETS; ++d) {
    a.Nd[d] = 0; a.NTd[d] = 0;
    if (d >= n_b || bt[d] == nullptr || Nd[d] <= 0) continue;
    MDSEG_REQUIRE(((uintptr_t)bt[d] & 15) == 0, "%s: B operand %d must be 16-byte aligned", who, d);
    const int NT = mdseg_head_tc16_tile(Nd[d]);
    const int n_tiles = (Nd[d] + NT - 1) / NT;
    a.Nd[d] = Nd[d]; a.NTd[d] = NT;
    tiles_max = n_tiles > tiles_max ? n_tiles : tiles_max;
    nt_max = NT > nt_max ? NT : nt_max;
    cuuint64_t dims[2] = {(cuuint64_t)ldb, (cuuint64_t)(n_tiles * NT)};
    cuuint64_t strides[1] = {(cuuint64_t)ldb * 2};
    cuuint32_t box[2] = {(cuuint32_t)kKB, (cuuint32_t)NT};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&mapsB.m[d], dt, 2, const_cast<void*>(bt[d]), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MDSEG_REQUIRE(r == CUDA_SUCCESS, "%s: cuTensorMapEncodeTiled failed for B operand %d (CUresult %d)", who, d, (int)r);
  }
  if (tiles_max == 0) return 0;
  const size_t smem = (size_t)kNStages * (kABytes + (size_t)nt_max * 128) + 1024;
  const dim3 grid((unsigned)tiles_max, (unsigned)((hw + kM - 1) / kM), (unsigned)n_images);
  // the variants in use: planar in and out; pixel-major x with planar fp32 y (forward); planar dy with a pixel-major
  // gradient (adjoint)
  MDSEG_REQUIRE(!(a_pm && out_pm) && (!a_pm || out_dtype == MDSEG_F32), "%s: unsupported layout combination", who);
#define MDSEG_H16_LAUNCH(TO, AK, PM) \
  do { if (launch_head16_kernel<TO, AK, PM>(mapA, mapsB, a, grid, smem, s)) return 1; } while (0)
  if (a_pm) MDSEG_H16_LAUNCH(float, true, false);
  else if (out_pm) {
    if (out_dtype == MDSEG_F32) MDSEG_H16_LAUNCH(float, false, true);
    else if (dtype == MDSEG_BF16) MDSEG_H16_LAUNCH(__nv_bfloat16, false, true);
    else MDSEG_H16_LAUNCH(__half, false, true);
  } else if (out_dtype == MDSEG_F32) MDSEG_H16_LAUNCH(float, false, false);
  else if (dtype == MDSEG_BF16) MDSEG_H16_LAUNCH(__nv_bfloat16, false, false);
  else MDSEG_H16_LAUNCH(__half, false, false);
#undef MDSEG_H16_LAUNCH
  MDSEG_LAUNCH_OK();
  return 0;
}
}  // namespace
}  // namespace mdseg

static bool layout_ok(int layout) { return layout == MDSEG_NCHW || layout == MDSEG_NHWC; }

extern "C" int mdseg_proj_fwd_tc16(const void* x, int dtype, int layout, int n_images, int C_uni, int64_t hw,
                                   const void* const* graphs_t, int ldb, const int* C_ds, int n_datasets,
                                   const int32_t* dataset_ids, float* y, int y_cmax, void* stream) {
  MDSEG_REQUIRE(layout_ok(layout), "mdseg_proj_fwd_tc16: layout %d is neither NCHW nor NHWC", layout);
  for (int d = 0; d < n_datasets && d < MDSEG_MAX_DATASETS; ++d)
    MDSEG_REQUIRE(!C_ds || C_ds[d] <= y_cmax, "mdseg_proj_fwd_tc16: y_cmax %d < C_ds %d", y_cmax, C_ds[d]);
  return mdseg::launch_head16(x, dtype, n_images, C_uni, hw, graphs_t, ldb, C_ds, n_datasets, dataset_ids, y, y_cmax, MDSEG_F32,
                              (cudaStream_t)stream, "mdseg_proj_fwd_tc16", 0, /*a_pm=*/layout == MDSEG_NHWC);
}

extern "C" int mdseg_proj_bwd_tc16(const void* dy16, int dtype, int layout, int n_images, int y_cmax, int64_t hw,
                                   const void* const* graphs_tt, int ldb, int C_uni, int n_datasets,
                                   const int32_t* dataset_ids, void* dx, int dx_dtype, void* stream) {
  MDSEG_REQUIRE(layout_ok(layout), "mdseg_proj_bwd_tc16: layout %d is neither NCHW nor NHWC", layout);
  MDSEG_REQUIRE(C_uni > 0 && n_datasets > 0 && n_datasets <= MDSEG_MAX_DATASETS, "mdseg_proj_bwd_tc16: bad shape");
  int Nd[MDSEG_MAX_DATASETS];
  for (int d = 0; d < n_datasets; ++d) Nd[d] = C_uni;
  return mdseg::launch_head16(dy16, dtype, n_images, y_cmax, hw, graphs_tt, ldb, Nd, n_datasets, dataset_ids, dx, C_uni,
                              dx_dtype, (cudaStream_t)stream, "mdseg_proj_bwd_tc16", /*zero_N=*/C_uni, /*a_pm=*/false,
                              /*out_pm=*/layout == MDSEG_NHWC);
}

// pixel slabs per image of the split-K d W GEMM: about two waves of CTAs, at least 4096 pixels per slab
static int dw_slabs_per_image(int n_images, int64_t hw, int tiles) {
  long long want = (2LL * 2 * mdseg::sm_count() + (long long)n_images * tiles - 1) / ((long long)n_images * tiles);
  const long long cap = (hw + 4095) / 4096;
  if (want > cap) want = cap;
  return (int)(want < 1 ? 1 : want);
}

// d W = dy16 x^T below contracts over the pixels: K = C_uni (channels of x), N = y_cmax (planes of dy16)
extern "C" size_t mdseg_proj_bwd_graph_tc16_workspace_bytes(int n_images, int K, int64_t hw, int N) {
  if (n_images <= 0 || K <= 0 || hw <= 0 || N <= 0) return 256;
  const int NT = mdseg_head_tc16_tile(K);
  const int n_tiles = (K + NT - 1) / NT, m_tiles = (N + 127) / 128;
  const int spi = dw_slabs_per_image(n_images, hw, m_tiles * n_tiles);
  return (size_t)n_images * spi * m_tiles * n_tiles * 128 * NT * 4 + 256;
}

// x planar [n_images, K, hw] is a K-major B operand like dy16; pixel-major [n_images, hw, K] (MDSEG_NHWC) an MN-major one
extern "C" int mdseg_proj_bwd_graph_tc16(const void* dy16, const void* x, int dtype, int layout, int n_images, int K,
                                         int64_t hw, int N, const int32_t* dataset_ids, int n_datasets, float* dW,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  using namespace mdseg;
  const bool x_pm = layout == MDSEG_NHWC;
  MDSEG_REQUIRE(layout_ok(layout), "mdseg_proj_bwd_graph_tc16: layout %d is neither NCHW nor NHWC", layout);
  MDSEG_REQUIRE(n_datasets > 0 && n_datasets <= MDSEG_MAX_DATASETS && (dataset_ids || n_datasets == 1),
                "mdseg_proj_bwd_graph_tc16: 1..%d datasets, dataset ids unless there is one", MDSEG_MAX_DATASETS);
  MDSEG_REQUIRE(dtype == MDSEG_BF16 || dtype == MDSEG_F16, "mdseg_proj_bwd_graph_tc16: operands must be bf16 or fp16");
  MDSEG_REQUIRE(n_images > 0 && n_images <= 65535 && K > 0 && N > 0 && hw > 0 && hw % 8 == 0,
                "mdseg_proj_bwd_graph_tc16: bad shape");
  MDSEG_REQUIRE(!x_pm || K % 8 == 0,
                "mdseg_proj_bwd_graph_tc16: the channel count must be a multiple of 8 (16-byte TMA pixel stride)");
  MDSEG_REQUIRE(dy16 && x && dW && workspace, "mdseg_proj_bwd_graph_tc16: null pointer");
  MDSEG_REQUIRE((((uintptr_t)dy16 | (uintptr_t)x) & 15) == 0, "mdseg_proj_bwd_graph_tc16: operands must be 16-byte aligned");
  MDSEG_REQUIRE(workspace_bytes >= mdseg_proj_bwd_graph_tc16_workspace_bytes(n_images, K, hw, N),
                "mdseg_proj_bwd_graph_tc16: workspace too small");
  const tma::EncodeTiledFn enc = tensor_map_encoder();
  if (enc == nullptr) return 1;
  DwArgs a;
  a.NT = mdseg_head_tc16_tile(K);
  a.n_tiles = (K + a.NT - 1) / a.NT;
  a.m_tiles = (N + 127) / 128;
  a.slabs_per_image = dw_slabs_per_image(n_images, hw, a.m_tiles * a.n_tiles);
  a.slab = ((hw + a.slabs_per_image - 1) / a.slabs_per_image + 63) / 64 * 64;
  a.slabs_per_image = (int)((hw + a.slab - 1) / a.slab);
  a.hw = hw;
  a.fmt = dtype == MDSEG_F16 ? 0 : 1;
  a.part = reinterpret_cast<float*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  const CUtensorMapDataType dt = dtype == MDSEG_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUtensorMap mapA, mapB;
  const cuuint32_t estr[3] = {1, 1, 1};
  {
    cuuint64_t dims[3] = {(cuuint64_t)hw, (cuuint64_t)N, (cuuint64_t)n_images};
    cuuint64_t strides[2] = {(cuuint64_t)hw * 2, (cuuint64_t)N * hw * 2};
    cuuint32_t box[3] = {64, 128, 1};
    CUresult r = enc(&mapA, dt, 3, const_cast<void*>(dy16), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MDSEG_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed for the gradient (CUresult %d)", (int)r);
  }
  {
    cuuint64_t dims[3] = {(cuuint64_t)hw, (cuuint64_t)K, (cuuint64_t)n_images};
    cuuint64_t strides[2] = {(cuuint64_t)hw * 2, (cuuint64_t)K * hw * 2};
    cuuint32_t box[3] = {64, (cuuint32_t)a.NT, 1};
    if (x_pm) {  // [n_images, hw, K]: boxes of [64 pixels][64 channels]
      dims[0] = (cuuint64_t)K; dims[1] = (cuuint64_t)hw;
      strides[0] = (cuuint64_t)K * 2;
      box[0] = 64; box[1] = 64;
    }
    CUresult r = enc(&mapB, dt, 3, const_cast<void*>(x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MDSEG_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed for the features (CUresult %d)", (int)r);
  }
  const int n_slabs_total = n_images * a.slabs_per_image;
  const size_t b_bytes = x_pm ? (size_t)((a.NT + 63) / 64) * 8192 : (size_t)a.NT * 128;
  const size_t smem = (size_t)kNStages * (128 * 128 + b_bytes) + 1024;
  cudaStream_t s = (cudaStream_t)stream;
  const dim3 grid((unsigned)(a.m_tiles * a.n_tiles), (unsigned)n_slabs_total);
  if (x_pm) {
    MDSEG_CUDA_OK(cudaFuncSetAttribute(head_tc16_dw_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    head_tc16_dw_kernel<true><<<grid, kThreads, smem, s>>>(mapA, mapB, a);
  } else {
    MDSEG_CUDA_OK(cudaFuncSetAttribute(head_tc16_dw_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    head_tc16_dw_kernel<false><<<grid, kThreads, smem, s>>>(mapA, mapB, a);
  }
  MDSEG_LAUNCH_OK();
  head_tc16_dw_reduce_kernel<<<dim3((unsigned)(((long long)N * K + 255) / 256), (unsigned)(dataset_ids ? n_datasets : 1)),
                               256, 0, s>>>(a, n_slabs_total, N, K, dataset_ids, dW);
  MDSEG_LAUNCH_OK();
  return 0;
}
