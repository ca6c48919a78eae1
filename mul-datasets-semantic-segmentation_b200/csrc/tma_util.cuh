// tma_util.cuh — the one copy of the mbarrier, bulk-copy, TMA (cp.async.bulk.tensor) and tcgen05 PTX wrappers every
// kernel file uses, packed-fp32 (FFMA2/FADD2) helpers and the host-side tensor-map builder of the warp-private fused
// kernels (up_ce_warp.cu, mds_bwd.cu).  sm_100a only.
#pragma once

#include <cuda.h>

#include "up_ce_internal.cuh"

namespace mdseg {
namespace tma {

struct alignas(64) Maps {
  CUtensorMap m[MDSEG_MAX_DATASETS];
};

#ifdef __CUDACC__
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "MDSEG_W_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra MDSEG_W_DONE;\n"
      "bra MDSEG_W_WAIT;\n"
      "MDSEG_W_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// 1-D bulk copy global -> shared, completion on an mbarrier (addresses and size multiples of 16 bytes)
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// tiled loads global -> shared, completion on an mbarrier.  Coordinates innermost first.
__device__ __forceinline__ void load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                        int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void prefetch_map(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}

// ---- tcgen05 (one CTA, cta_group::1) ----
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// arrive on `bar` when every MMA issued so far by this thread has retired
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T, 16-bit inputs, fp32 accumulate
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// 16 consecutive 32-bit columns of this thread's TMEM lane.  The registers are valid only after a tmem_wait_ld.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
// wait for this thread's outstanding TMEM loads
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// the same wait, naming the registers it releases, so that the compiler cannot move a use of r above it
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :: "memory");
}
// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, version 1).  `sbo` = bytes between 8-row groups,
// `lbo` = bytes between the core matrices adjacent in the leading dimension.
enum UmmaLayout : uint64_t { kNoSwizzle = 0, kSwizzle128B = 2 };
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, UmmaLayout layout) {
  return (uint64_t)((saddr & 0x3ffffu) >> 4) | ((uint64_t)((lbo >> 4) & 0x3fffu) << 16) |
         ((uint64_t)((sbo >> 4) & 0x3fffu) << 32) | (1ull << 46) | ((uint64_t)layout << 61);
}

// ---- packed fp32 pairs: one issue slot for two lanes of work (FFMA2 / FADD2 / FMUL2 on sm_100) ----
__device__ __forceinline__ unsigned long long pk(float2 a) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a.x), "f"(a.y));
  return r;
}
__device__ __forceinline__ float2 upk(unsigned long long r) {
  float2 a;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a.x), "=f"(a.y) : "l"(r));
  return a;
}
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(pk(a)), "l"(pk(b)), "l"(pk(c)));
  return upk(d);
}
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  unsigned long long d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk(a)), "l"(pk(b)));
  return upk(d);
}
__device__ __forceinline__ float2 sub2(float2 a, float2 b) {
  unsigned long long d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk(a)), "l"(pk(b)));
  return upk(d);
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
  unsigned long long d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk(a)), "l"(pk(b)));
  return upk(d);
}
__device__ __forceinline__ float2 dup2(float a) { return make_float2(a, a); }
// class id as a pair of fp16 values (compared against two pixels' labels at once): the id of class c + 1 from the id
// of class c by one packed half add (exact below 2048) instead of an int -> half conversion on the XU pipe per class
__device__ __forceinline__ uint32_t class_pair(int c) {
  const uint32_t ch = (uint32_t)__half_as_ushort(__int2half_rn(c));
  return ch | (ch << 16);
}
__device__ __forceinline__ uint32_t next_class2(uint32_t c2) {
  asm("add.f16x2 %0, %0, %1;" : "+r"(c2) : "r"(0x3c003c00u));
  return c2;
}
__device__ __forceinline__ float2 ex2_2(float2 a) { return make_float2(ex2_approx(a.x), ex2_approx(a.y)); }


// align_corners=True source position of destination index `dst` expressed as (cell, lambda) with
// cell in [0, n_in-2]: the last source index is folded into the last cell with lambda = 1, which
// gives exactly ATen's value (i1 = i0 there, weights sum to 1) and makes every cell regular.
__device__ __forceinline__ void axis_cell(const AxisMap& m, int dst, int& cell, float& lam) {
  const float s = m.scale * (float)dst;
  const int i0 = (int)s;
  if (i0 >= m.n_in - 1) {
    cell = m.n_in - 2;
    lam = 1.0f;
  } else {
    cell = i0;
    lam = s - (float)i0;
  }
}
// label range [beg, end) of cell `c` along an axis with n_out destinations
__device__ __forceinline__ void cell_span(const AxisMap& m, int c, int n_out, int& beg, int& end) {
  beg = first_dst_ge(m, c, n_out);
  end = (c >= m.n_in - 2) ? n_out : first_dst_ge(m, c + 1, n_out);
}
#endif  // __CUDACC__

// host: the driver's cuTensorMapEncodeTiled, looked up once; NULL when the driver does not have it
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn();
// host: make the primary context current on the calling thread before a driver entry point is called (autograd runs
// the backward on its own thread, where only runtime calls were made).  0 = OK, else set_error was called.
int bind_primary_context();
// host: tensor maps over the fp32 sources [n_images][C_alloc][h][w] with box (box_w, box_h, box_c, 1)
int make_maps(const mdseg_src_table& src, const Geom& gm, int n_images, int box_w, int box_h, int box_c, Maps* out);
// cmax[b, y, x] = max_c src[b, c, y, x] for fp32 sources with hw % 4 == 0 (src.cmax is the output plane)
int channel_max(const mdseg_src_table& src, const int32_t* dataset_ids, int n_images, int64_t hw, cudaStream_t s);
// fast-path geometry: fp32 sources, 16-byte aligned rows, h,w >= 2, 1 <= up-sampling factor <= 5, C <= 254
bool fast_geometry(const mdseg_src_table& src, const Geom& gm);

}  // namespace tma
}  // namespace mdseg
