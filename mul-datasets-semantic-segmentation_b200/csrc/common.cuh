// common.cuh — shared device/host helpers for libmdseg_b200 (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mdseg.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libmdseg_b200 is written for sm_100a (B200) only"
#endif

namespace mdseg {

// ---- host side -----------------------------------------------------------
void set_error(const char* fmt, ...);
int sm_count();

#define MDSEG_CUDA_OK(expr)                                                   \
  do {                                                                        \
    cudaError_t _e = (expr);                                                  \
    if (_e != cudaSuccess) {                                                  \
      ::mdseg::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,        \
                         cudaGetErrorString(_e));                             \
      return 1;                                                               \
    }                                                                         \
  } while (0)

#define MDSEG_REQUIRE(cond, ...)                                              \
  do {                                                                        \
    if (!(cond)) {                                                            \
      ::mdseg::set_error(__VA_ARGS__);                                        \
      return 2;                                                               \
    }                                                                         \
  } while (0)

#define MDSEG_LAUNCH_OK()                                                     \
  do {                                                                        \
    cudaError_t _e = cudaGetLastError();                                      \
    if (_e != cudaSuccess) {                                                  \
      ::mdseg::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__,    \
                         cudaGetErrorString(_e));                             \
      return 1;                                                               \
    }                                                                         \
  } while (0)

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline bool is_float_dtype(int d) { return d == MDSEG_F32 || d == MDSEG_BF16 || d == MDSEG_F16; }
static inline bool is_int_dtype(int d) { return d == MDSEG_U8 || d == MDSEG_I32 || d == MDSEG_I64; }
static inline int dtype_size(int d) {
  switch (d) {
    case MDSEG_F32: return 4;
    case MDSEG_BF16: return 2;
    case MDSEG_F16: return 2;
    case MDSEG_U8: return 1;
    case MDSEG_I32: return 4;
    case MDSEG_I64: return 8;
  }
  return 0;
}

// Type dispatch of a dtype code: f(type_tag<T>{}) for the C++ type T the code names, or error 2 naming the entry
// point (who) and the parameter (what) for a code outside the set.
template <typename T> struct type_tag { using type = T; };

template <typename F>
inline int with_float_type(int code, const char* who, const char* what, F&& f) {
  switch (code) {
    case MDSEG_F32: return f(type_tag<float>{});
    case MDSEG_BF16: return f(type_tag<__nv_bfloat16>{});
    case MDSEG_F16: return f(type_tag<__half>{});
  }
  set_error("%s: unsupported %s %d", who, what, code);
  return 2;
}

template <typename F>
inline int with_int_type(int code, const char* who, const char* what, F&& f) {
  switch (code) {
    case MDSEG_U8: return f(type_tag<uint8_t>{});
    case MDSEG_I32: return f(type_tag<int32_t>{});
    case MDSEG_I64: return f(type_tag<int64_t>{});
  }
  set_error("%s: unsupported %s %d", who, what, code);
  return 2;
}

// Source tables: 1..MDSEG_MAX_DATASETS datasets ...
inline bool src_count_ok(const mdseg_src_table* s) {
  return s && s->n_datasets > 0 && s->n_datasets <= MDSEG_MAX_DATASETS;
}
// ... each with classes and a base pointer.
inline int check_src(const mdseg_src_table* s, const char* who) {
  MDSEG_REQUIRE(src_count_ok(s), "%s: bad source table", who);
  for (int i = 0; i < s->n_datasets; ++i)
    MDSEG_REQUIRE(s->C[i] > 0 && s->base[i] != nullptr, "%s: dataset %d has no source", who, i);
  return 0;
}
// the widest class count of a source table
inline int max_c(const mdseg_src_table* s) {
  int m = 0;
  for (int i = 0; i < s->n_datasets; ++i) m = s->C[i] > m ? s->C[i] : m;
  return m;
}

// Graph tables: 1..MDSEG_MAX_DATASETS datasets onto C_uni > 0 unified classes.
inline bool graph_header_ok(const mdseg_graph_table* t) {
  return t && t->n_datasets > 0 && t->n_datasets <= MDSEG_MAX_DATASETS && t->C_uni > 0;
}
// the widest dataset class count C_ds of a graph table
inline int max_c_ds(const mdseg_graph_table* t) {
  int m = 0;
  for (int i = 0; i < t->n_datasets; ++i) m = t->g[i].C_ds > m ? t->g[i].C_ds : m;
  return m;
}

// The adjoint of a bilinear up-sampling writes the two vertical taps of every low-resolution cell into two fp32 planes
// per dataset, A_d and B_d, each [n_images, C_d, h, w]; the gradient is their sum.  Bytes of that workspace:
inline size_t two_plane_bytes(const mdseg_src_table* src, int n_images, int h, int w) {
  size_t planes = 0;
  for (int i = 0; i < src->n_datasets; ++i) planes += 2 * (size_t)n_images * src->C[i] * h * w * 4;
  return planes + 256;
}
// Carves [A_d, B_d] out of the workspace, zeroes them when `zero`, runs adjoint(dA, dB) on the fp32 tables of the
// planes and adds every pair into dst (dense [n_images, C_d, h, w] tensors of dst->dtype).
template <typename Adjoint>
int two_plane_adjoint(const char* who, const mdseg_src_table* src, const mdseg_src_table* dst, int n_images, int h,
                      int w, void* workspace, bool zero, cudaStream_t s, Adjoint&& adjoint) {
  const int64_t hw = (int64_t)h * w;
  float* ws = reinterpret_cast<float*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  mdseg_src_table dA = *src, dB = *src;
  dA.dtype = MDSEG_F32; dB.dtype = MDSEG_F32; dA.cmax = nullptr; dB.cmax = nullptr;
  size_t off = 0;
  for (int i = 0; i < src->n_datasets; ++i) {
    const size_t n = (size_t)n_images * src->C[i] * hw;
    dA.base[i] = ws + off; dB.base[i] = ws + off + n;
    dA.image_stride[i] = (long long)src->C[i] * hw; dB.image_stride[i] = dA.image_stride[i];
    dA.C_alloc[i] = src->C[i]; dB.C_alloc[i] = src->C[i];
    off += 2 * n;
  }
  if (zero) MDSEG_CUDA_OK(cudaMemsetAsync(ws, 0, off * 4, s));
  if (int rc = adjoint(dA, dB)) return rc;
  for (int i = 0; i < src->n_datasets; ++i) {
    MDSEG_REQUIRE(dst->image_stride[i] == (long long)src->C[i] * hw,
                  "%s: the two-plane route needs dense [n_images, C, h, w] destinations", who);
    if (int rc = mdseg_add_planes((const float*)dA.base[i], (const float*)dB.base[i], const_cast<void*>(dst->base[i]),
                                  dst->dtype, (int64_t)n_images * src->C[i] * hw, s))
      return rc;
  }
  return 0;
}

// ---- device side ---------------------------------------------------------
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }

// Streaming (read-once) loads: keep them out of L1 so resident tiles survive.
__device__ __forceinline__ int4 ldg_stream_v4(const void* p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ int2 ldg_stream_v2(const void* p) {
  int2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.s32 {%0,%1}, [%2];"
               : "=r"(r.x), "=r"(r.y)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_stream_v4(void* p, int4 v) {
  asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p),
               "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}

// Load V consecutive elements of type T (V*sizeof(T) is 4, 8 or 16 bytes,
// pointer aligned accordingly) and widen to fp32.
template <typename T, int V> struct VecLoad;
// raw(): the load alone (what is kept in registers while several loads are in flight); unpack(): raw -> fp32
template <> struct VecLoad<float, 4> {
  using Raw = int4;
  static __device__ __forceinline__ Raw raw(const float* p) { return ldg_stream_v4(p); }
  static __device__ __forceinline__ void unpack(const Raw& r, float (&o)[4]) {
    o[0] = __int_as_float(r.x); o[1] = __int_as_float(r.y);
    o[2] = __int_as_float(r.z); o[3] = __int_as_float(r.w);
  }
  static __device__ __forceinline__ void load(const float* p, float (&o)[4]) { unpack(raw(p), o); }
  static __device__ __forceinline__ void store(float* p, const float (&v)[4]) {
    int4 r = make_int4(__float_as_int(v[0]), __float_as_int(v[1]),
                       __float_as_int(v[2]), __float_as_int(v[3]));
    stg_stream_v4(p, r);
  }
};
template <> struct VecLoad<float, 1> {
  using Raw = float;
  static __device__ __forceinline__ Raw raw(const float* p) { return __ldg(p); }
  static __device__ __forceinline__ void unpack(const Raw& r, float (&o)[1]) { o[0] = r; }
  static __device__ __forceinline__ void load(const float* p, float (&o)[1]) { o[0] = __ldg(p); }
  static __device__ __forceinline__ void store(float* p, const float (&v)[1]) { p[0] = v[0]; }
};
template <> struct VecLoad<__nv_bfloat16, 8> {
  using Raw = int4;
  static __device__ __forceinline__ Raw raw(const __nv_bfloat16* p) { return ldg_stream_v4(p); }
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&o)[8]) { unpack(raw(p), o); }
  static __device__ __forceinline__ void unpack(const Raw& r, float (&o)[8]) {
    const uint32_t w[4] = {(uint32_t)r.x, (uint32_t)r.y, (uint32_t)r.z, (uint32_t)r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      o[2 * i] = __uint_as_float(w[i] << 16);
      o[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&t);
    }
    stg_stream_v4(p, make_int4((int)w[0], (int)w[1], (int)w[2], (int)w[3]));
  }
};
// four 16-bit values per 8-byte load: the forward of the full-resolution CE keeps 8 planes x 4 pixels in registers
// (8 planes x 8 pixels cost 157 registers and one resident CTA per SM)
template <> struct VecLoad<__nv_bfloat16, 4> {
  using Raw = int2;
  static __device__ __forceinline__ Raw raw(const __nv_bfloat16* p) { return ldg_stream_v2(p); }
  static __device__ __forceinline__ void unpack(const Raw& r, float (&o)[4]) {
    const uint32_t w[2] = {(uint32_t)r.x, (uint32_t)r.y};
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      o[2 * i] = __uint_as_float(w[i] << 16);
      o[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&o)[4]) { unpack(raw(p), o); }
};
template <> struct VecLoad<__half, 4> {
  using Raw = int2;
  static __device__ __forceinline__ Raw raw(const __half* p) { return ldg_stream_v2(p); }
  static __device__ __forceinline__ void unpack(const Raw& r, float (&o)[4]) {
    const uint32_t w[2] = {(uint32_t)r.x, (uint32_t)r.y};
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
      o[2 * i] = f.x; o[2 * i + 1] = f.y;
    }
  }
  static __device__ __forceinline__ void load(const __half* p, float (&o)[4]) { unpack(raw(p), o); }
};
template <> struct VecLoad<__nv_bfloat16, 1> {
  using Raw = __nv_bfloat16;
  static __device__ __forceinline__ Raw raw(const __nv_bfloat16* p) { return *p; }
  static __device__ __forceinline__ void unpack(const Raw& r, float (&o)[1]) { o[0] = __bfloat162float(r); }
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&o)[1]) { o[0] = __bfloat162float(*p); }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[1]) { p[0] = __float2bfloat16_rn(v[0]); }
};
template <> struct VecLoad<__half, 8> {
  using Raw = int4;
  static __device__ __forceinline__ Raw raw(const __half* p) { return ldg_stream_v4(p); }
  static __device__ __forceinline__ void load(const __half* p, float (&o)[8]) { unpack(raw(p), o); }
  static __device__ __forceinline__ void unpack(const Raw& r, float (&o)[8]) {
    const uint32_t w[4] = {(uint32_t)r.x, (uint32_t)r.y, (uint32_t)r.z, (uint32_t)r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __half2 t = *reinterpret_cast<const __half2*>(&w[i]);
      float2 f = __half22float2(t);
      o[2 * i] = f.x; o[2 * i + 1] = f.y;
    }
  }
  static __device__ __forceinline__ void store(__half* p, const float (&v)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __half2 t = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&t);
    }
    stg_stream_v4(p, make_int4((int)w[0], (int)w[1], (int)w[2], (int)w[3]));
  }
};
template <> struct VecLoad<__half, 1> {
  using Raw = __half;
  static __device__ __forceinline__ Raw raw(const __half* p) { return *p; }
  static __device__ __forceinline__ void unpack(const Raw& r, float (&o)[1]) { o[0] = __half2float(r); }
  static __device__ __forceinline__ void load(const __half* p, float (&o)[1]) { o[0] = __half2float(*p); }
  static __device__ __forceinline__ void store(__half* p, const float (&v)[1]) { p[0] = __float2half_rn(v[0]); }
};

// Labels: read one label as int (u8 / i32 / i64 sources).
template <typename L> __device__ __forceinline__ int load_label(const L* p, int64_t i) { return (int)p[i]; }
template <> __device__ __forceinline__ int load_label<int64_t>(const int64_t* p, int64_t i) {
  long long v = p[i];
  // clamp to int range keeping "out of range" detectable
  return (v < -1 || v > 0x7fffffffLL) ? -1 : (int)v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ unsigned warp_sum(unsigned v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block-level accumulation of the three OHEM statistics into a state:
// one 64-bit atomic per counter per CTA.
__device__ __forceinline__ void block_accumulate_stats(mdseg_ohem_state* st, unsigned n_valid,
                                                       unsigned n_hard, double sum_hard,
                                                       unsigned n_px) {
  __shared__ unsigned s_valid, s_hard, s_px;
  __shared__ double s_sum;
  if (threadIdx.x == 0) { s_valid = 0; s_hard = 0; s_px = 0; s_sum = 0.0; }
  __syncthreads();
  n_valid = warp_sum(n_valid);
  n_hard = warp_sum(n_hard);
  n_px = warp_sum(n_px);
  sum_hard = warp_sum(sum_hard);
  if ((threadIdx.x & 31) == 0) {
    if (n_valid) atomicAdd(&s_valid, n_valid);
    if (n_hard) atomicAdd(&s_hard, n_hard);
    if (n_px) atomicAdd(&s_px, n_px);
    if (n_hard) atomicAdd(&s_sum, sum_hard);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_valid) atomicAdd(&st->n_valid, (unsigned long long)s_valid);
    if (s_hard) { atomicAdd(&st->n_hard, (unsigned long long)s_hard); atomicAdd(&st->sum_hard, s_sum); }
    if (s_px) atomicAdd(&st->n_px, (unsigned long long)s_px);
  }
}

// Order-preserving map float -> uint32 (larger float <-> larger key).
__device__ __forceinline__ uint32_t float_key(float f) {
  uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_float(uint32_t k) {
  uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(b);
}

// align_corners=True source coordinate, exactly as ATen computes it in fp32
// (area_pixel_compute_source_index with align_corners: scale * dst).
struct AxisMap {
  float scale;  // (in-1)/(out-1), 0 when out == 1
  int n_in;
  __device__ __forceinline__ void at(int dst, int& i0, int& i1, float& l0, float& l1) const {
    float s = scale * (float)dst;
    i0 = (int)s;
    if (i0 > n_in - 1) i0 = n_in - 1;  // guards fp rounding at the last index
    i1 = i0 + ((i0 < n_in - 1) ? 1 : 0);
    l1 = s - (float)i0;
    l0 = 1.0f - l1;
  }
  __device__ __forceinline__ int floor_at(int dst) const {
    int i0 = (int)(scale * (float)dst);
    return i0 > n_in - 1 ? n_in - 1 : i0;
  }
};
static inline float axis_scale(int n_in, int n_out) {
  return n_out > 1 ? (float)(n_in - 1) / (float)(n_out - 1) : 0.0f;
}

}  // namespace mdseg
