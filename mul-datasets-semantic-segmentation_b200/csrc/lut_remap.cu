// lut_remap.cu — 256-entry label LUT gather (SURVEY §8 rows a1/a2).
//
// Reference work replaced:
//   label = self.lb_map[label]                      lib/base_dataset.py:81-82
//   mask[labels==k] = v[j] for every (k, v)         lib/class_remap.py:39-48,55-64
//   Remap_pred[preds==lb] = k                       lib/class_remap.py:189-203
// Each of these is out[p] = lut[in[p]] with a uint8[256] table; values outside
// [0,255] (only possible for int32/int64 inputs) map to `oob`.
//
// HBM-bound byte kernel: 16 elements per thread per iteration, 128-bit
// loads/stores on both sides, LUT staged once per CTA in shared memory.
// Algorithmic bytes per pixel: sizeof(in) + sizeof(out).
#include "common.cuh"

namespace mdseg {
namespace {

constexpr int kE = 16;  // elements per thread per iteration

template <typename T> struct Pack16;

template <> struct Pack16<uint8_t> {
  static constexpr int kVecs = 1;
  static __device__ __forceinline__ void unpack(const int4* v, int (&x)[kE]) {
    const uint32_t w[4] = {(uint32_t)v[0].x, (uint32_t)v[0].y, (uint32_t)v[0].z, (uint32_t)v[0].w};
#pragma unroll
    for (int i = 0; i < kE; ++i) x[i] = (w[i >> 2] >> (8 * (i & 3))) & 0xff;
  }
  static __device__ __forceinline__ void pack(const int (&x)[kE], int4* v) {
    uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
    for (int i = 0; i < kE; ++i) w[i >> 2] |= ((uint32_t)x[i] & 0xffu) << (8 * (i & 3));
    v[0] = make_int4((int)w[0], (int)w[1], (int)w[2], (int)w[3]);
  }
};
template <> struct Pack16<int32_t> {
  static constexpr int kVecs = 4;
  static __device__ __forceinline__ void unpack(const int4* v, int (&x)[kE]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int a = v[j].x, b = v[j].y, c = v[j].z, d = v[j].w;
      x[4 * j + 0] = ((unsigned)a < 256u) ? a : -1;
      x[4 * j + 1] = ((unsigned)b < 256u) ? b : -1;
      x[4 * j + 2] = ((unsigned)c < 256u) ? c : -1;
      x[4 * j + 3] = ((unsigned)d < 256u) ? d : -1;
    }
  }
  static __device__ __forceinline__ void pack(const int (&x)[kE], int4* v) {
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = make_int4(x[4 * j], x[4 * j + 1], x[4 * j + 2], x[4 * j + 3]);
  }
};
template <> struct Pack16<int64_t> {
  static constexpr int kVecs = 8;
  static __device__ __forceinline__ void unpack(const int4* v, int (&x)[kE]) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      x[2 * j + 0] = (v[j].y == 0 && (unsigned)v[j].x < 256u) ? v[j].x : -1;
      x[2 * j + 1] = (v[j].w == 0 && (unsigned)v[j].z < 256u) ? v[j].z : -1;
    }
  }
  static __device__ __forceinline__ void pack(const int (&x)[kE], int4* v) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      v[j] = make_int4(x[2 * j], x[2 * j] >> 31, x[2 * j + 1], x[2 * j + 1] >> 31);
  }
};

// blockIdx.y = image: `n` elements per image; image b uses table lut + 256 * lut_ids[b] (lut_ids NULL: table 0).
// An id outside [0, n_luts) maps the whole image to `oob` and raises MDSEG_ERR_DATASET_ID.
template <typename In, typename Out>
__global__ void __launch_bounds__(256) lut_remap_kernel(const In* __restrict__ in, Out* __restrict__ out,
                                                       const uint8_t* __restrict__ lut, int oob, int64_t n,
                                                       const int32_t* __restrict__ lut_ids, int n_luts,
                                                       int* err_flag) {
  __shared__ uint8_t s_lut[256];
  {
    const int id = lut_ids ? lut_ids[blockIdx.y] : 0;
    const bool ok = id >= 0 && id < n_luts;
    s_lut[threadIdx.x] = ok ? lut[(int64_t)id * 256 + threadIdx.x] : (uint8_t)oob;
    if (!ok && threadIdx.x == 0 && blockIdx.x == 0 && err_flag) atomicOr(err_flag, MDSEG_ERR_DATASET_ID);
    in += (int64_t)blockIdx.y * n;
    out += (int64_t)blockIdx.y * n;
  }
  __syncthreads();

  const int64_t nvec = n / kE;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += stride) {
    int4 a[Pack16<In>::kVecs];
    const int4* src = reinterpret_cast<const int4*>(in + v * kE);
#pragma unroll
    for (int j = 0; j < Pack16<In>::kVecs; ++j) a[j] = ldg_stream_v4(src + j);
    int x[kE];
    Pack16<In>::unpack(a, x);
#pragma unroll
    for (int i = 0; i < kE; ++i) x[i] = (x[i] >= 0) ? (int)s_lut[x[i]] : oob;
    int4 o[Pack16<Out>::kVecs];
    Pack16<Out>::pack(x, o);
    int4* dst = reinterpret_cast<int4*>(out + v * kE);
#pragma unroll
    for (int j = 0; j < Pack16<Out>::kVecs; ++j) stg_stream_v4(dst + j, o[j]);
  }
  // ragged tail (< 16 elements)
  const int64_t t0 = nvec * kE + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t0 < n) {
    long long xv = (long long)in[t0];
    out[t0] = (Out)((xv >= 0 && xv < 256) ? (int)s_lut[xv] : oob);
  }
}

// Coalesced on BOTH sides for any (In, Out) width pair: a warp owns a tile of 512 consecutive pixels,
// loads it with 16-byte vectors in the input's own coalesced order, looks the bytes up and parks them in a
// 512-byte shared-memory tile, then re-reads that tile in the output's coalesced order and stores 16-byte
// vectors.  (The thread-contiguous variant above writes 128-byte runs per thread when widening u8 -> i64:
// every store instruction touches 32 different lines.)
template <typename T> struct Lane16 {           // pixels one lane moves per 16-byte vector
  static constexpr int kPx = 16 / (int)sizeof(T);
};
template <typename In> __device__ __forceinline__ int in_value(const int4& v, int i);
template <> __device__ __forceinline__ int in_value<uint8_t>(const int4& v, int i) {
  const uint32_t w = i < 4 ? (uint32_t)v.x : i < 8 ? (uint32_t)v.y : i < 12 ? (uint32_t)v.z : (uint32_t)v.w;
  return (int)((w >> (8 * (i & 3))) & 0xffu);
}
template <> __device__ __forceinline__ int in_value<int32_t>(const int4& v, int i) {
  const int a = i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w;
  return ((unsigned)a < 256u) ? a : -1;
}
template <> __device__ __forceinline__ int in_value<int64_t>(const int4& v, int i) {
  const int lo = i == 0 ? v.x : v.z, hi = i == 0 ? v.y : v.w;
  return (hi == 0 && (unsigned)lo < 256u) ? lo : -1;
}
template <typename Out> __device__ __forceinline__ int4 out_pack(const uint8_t* t);  // t: Lane16<Out>::kPx bytes
template <> __device__ __forceinline__ int4 out_pack<uint8_t>(const uint8_t* t) {
  return *reinterpret_cast<const int4*>(t);
}
template <> __device__ __forceinline__ int4 out_pack<int32_t>(const uint8_t* t) {
  const uint32_t w = *reinterpret_cast<const uint32_t*>(t);
  return make_int4((int)(w & 0xff), (int)((w >> 8) & 0xff), (int)((w >> 16) & 0xff), (int)(w >> 24));
}
template <> __device__ __forceinline__ int4 out_pack<int64_t>(const uint8_t* t) {
  const uint32_t w = *reinterpret_cast<const uint16_t*>(t);
  return make_int4((int)(w & 0xff), 0, (int)(w >> 8), 0);
}

template <typename In, typename Out>
__global__ void __launch_bounds__(256) lut_remap_tile_kernel(const In* __restrict__ in, Out* __restrict__ out,
                                                            const uint8_t* __restrict__ lut, int oob, int64_t n,
                                                            const int32_t* __restrict__ lut_ids, int n_luts,
                                                            int* err_flag) {
  constexpr int kTile = 512;
  __shared__ uint8_t s_lut[256];
  __shared__ __align__(16) uint8_t s_tile[8][kTile];
  {
    const int id = lut_ids ? lut_ids[blockIdx.y] : 0;
    const bool ok = id >= 0 && id < n_luts;
    s_lut[threadIdx.x] = ok ? lut[(int64_t)id * 256 + threadIdx.x] : (uint8_t)oob;
    if (!ok && threadIdx.x == 0 && blockIdx.x == 0 && err_flag) atomicOr(err_flag, MDSEG_ERR_DATASET_ID);
    in += (int64_t)blockIdx.y * n;
    out += (int64_t)blockIdx.y * n;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t* tile = s_tile[warp];
  constexpr int kIn = Lane16<In>::kPx, kOut = Lane16<Out>::kPx;
  constexpr int kInIt = kTile / (32 * kIn), kOutIt = kTile / (32 * kOut);
  const int64_t n_tiles = n / kTile;
  const int64_t wstride = (int64_t)gridDim.x * 8;
  for (int64_t t = (int64_t)blockIdx.x * 8 + warp; t < n_tiles; t += wstride) {
    const In* src = in + t * kTile;
    int4 v[kInIt];
#pragma unroll
    for (int j = 0; j < kInIt; ++j) v[j] = ldg_stream_v4(src + (j * 32 + lane) * kIn);
#pragma unroll
    for (int j = 0; j < kInIt; ++j) {
      uint8_t o[kIn];
#pragma unroll
      for (int i = 0; i < kIn; ++i) {
        const int x = in_value<In>(v[j], i);
        o[i] = (uint8_t)((x >= 0) ? (int)s_lut[x] : oob);
      }
      uint8_t* dst = tile + (j * 32 + lane) * kIn;
      if (kIn == 16) {
        uint32_t w[4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
          w[q] = o[4 * q] | ((uint32_t)o[4 * q + 1] << 8) | ((uint32_t)o[4 * q + 2] << 16) | ((uint32_t)o[4 * q + 3] << 24);
        *reinterpret_cast<int4*>(dst) = make_int4((int)w[0], (int)w[1], (int)w[2], (int)w[3]);
      } else if (kIn == 4) {
        *reinterpret_cast<uint32_t*>(dst) = o[0] | ((uint32_t)o[1] << 8) | ((uint32_t)o[2] << 16) | ((uint32_t)o[3] << 24);
      } else {
        *reinterpret_cast<uint16_t*>(dst) = (uint16_t)(o[0] | ((uint16_t)o[1] << 8));
      }
    }
    __syncwarp();
    Out* dstg = out + t * kTile;
#pragma unroll
    for (int j = 0; j < kOutIt; ++j)
      stg_stream_v4(dstg + (j * 32 + lane) * kOut, out_pack<Out>(tile + (j * 32 + lane) * kOut));
    __syncwarp();
  }
  // ragged tail (< 512 elements)
  for (int64_t i = n_tiles * kTile + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    long long xv = (long long)in[i];
    out[i] = (Out)((xv >= 0 && xv < 256) ? (int)s_lut[xv] : oob);
  }
}

// Unaligned fallback: one element per thread.
template <typename In, typename Out>
__global__ void __launch_bounds__(256) lut_remap_scalar_kernel(const In* __restrict__ in, Out* __restrict__ out,
                                                              const uint8_t* __restrict__ lut, int oob, int64_t n,
                                                              const int32_t* __restrict__ lut_ids, int n_luts,
                                                              int* err_flag) {
  __shared__ uint8_t s_lut[256];
  {
    const int id = lut_ids ? lut_ids[blockIdx.y] : 0;
    const bool ok = id >= 0 && id < n_luts;
    s_lut[threadIdx.x] = ok ? lut[(int64_t)id * 256 + threadIdx.x] : (uint8_t)oob;
    if (!ok && threadIdx.x == 0 && blockIdx.x == 0 && err_flag) atomicOr(err_flag, MDSEG_ERR_DATASET_ID);
    in += (int64_t)blockIdx.y * n;
    out += (int64_t)blockIdx.y * n;
  }
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    long long xv = (long long)in[i];
    out[i] = (Out)((xv >= 0 && xv < 256) ? (int)s_lut[xv] : oob);
  }
}

template <typename In, typename Out>
int launch(const void* in, void* out, const uint8_t* lut, int oob, int64_t n, cudaStream_t st,
           const int32_t* lut_ids = nullptr, int n_luts = 1, int n_images = 1, int* err_flag = nullptr) {
  if (n == 0 || n_images == 0) return 0;
  // per-image slices keep the 16-byte alignment only when the image size is a multiple of 16 elements
  const bool aligned = (((uintptr_t)in | (uintptr_t)out) & 15) == 0 && (n_images == 1 || n % kE == 0);
  const int sms = sm_count();
  const int64_t cap = ceil_div64((int64_t)sms * 8, n_images);
  if (aligned) {
    int64_t nvec = n / kE;
    int64_t blocks = ceil_div64(nvec > 0 ? nvec : 1, 256);
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    if (sizeof(In) != sizeof(Out))  // widening / narrowing: the tile kernel keeps both sides coalesced
      lut_remap_tile_kernel<In, Out><<<dim3((unsigned)blocks, (unsigned)n_images), 256, 0, st>>>(
          (const In*)in, (Out*)out, lut, oob, n, lut_ids, n_luts, err_flag);
    else
      lut_remap_kernel<In, Out><<<dim3((unsigned)blocks, (unsigned)n_images), 256, 0, st>>>(
          (const In*)in, (Out*)out, lut, oob, n, lut_ids, n_luts, err_flag);
  } else {
    int64_t blocks = ceil_div64(n, 256);
    if (blocks > cap) blocks = cap;
    lut_remap_scalar_kernel<In, Out><<<dim3((unsigned)blocks, (unsigned)n_images), 256, 0, st>>>(
        (const In*)in, (Out*)out, lut, oob, n, lut_ids, n_luts, err_flag);
  }
  MDSEG_LAUNCH_OK();
  return 0;
}

}  // namespace
}  // namespace mdseg

extern "C" int mdseg_lut_remap(const void* in, int in_dtype, void* out, int out_dtype, const uint8_t* lut256,
                               int oob, int64_t n, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(n >= 0, "mdseg_lut_remap: n < 0");
  MDSEG_REQUIRE(n == 0 || (in && out && lut256), "mdseg_lut_remap: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  return with_int_type(in_dtype, "mdseg_lut_remap", "in_dtype", [&](auto i) {
    return with_int_type(out_dtype, "mdseg_lut_remap", "out_dtype", [&](auto o) {
      return launch<typename decltype(i)::type, typename decltype(o)::type>(in, out, lut256, oob, n, st);
    });
  });
}

extern "C" int mdseg_lut_remap_images(const void* in, int in_dtype, void* out, int out_dtype, const uint8_t* luts,
                                      int n_luts, const int32_t* lut_ids, int oob, int n_images,
                                      int64_t px_per_image, int32_t* err_flag, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && px_per_image >= 0 && n_luts > 0,
                "mdseg_lut_remap_images: bad shape");
  if (n_images == 0 || px_per_image == 0) return 0;
  MDSEG_REQUIRE(in && out && luts, "mdseg_lut_remap_images: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  return with_int_type(in_dtype, "mdseg_lut_remap_images", "in_dtype", [&](auto i) {
    return with_int_type(out_dtype, "mdseg_lut_remap_images", "out_dtype", [&](auto o) {
      return launch<typename decltype(i)::type, typename decltype(o)::type>(in, out, luts, oob, px_per_image, st,
                                                                            lut_ids, n_luts, n_images, err_flag);
    });
  });
}
