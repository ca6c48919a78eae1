// multihot.cu — multi-hot label remap (SURVEY §8 row a4).
//
// Reference work replaced (lib/class_remap.py:239-276, ClassRemapOneHotLabel):
//   outMultiLabels = zeros([b, h, w, C_uni], bool)
//   for k, v in remap.items(): outMultiLabels[labels == k, v] = 1          (SegRemapping)
//   ... only classes with a single target                                   (SingleSegRemappingOneHot)
// i.e. one compare + masked scatter per dataset class.  Both are out[p, :] = table[labels[p], :] with a
// [256, C_uni] 0/1 table built once from the class_remap dict; labels outside [0, 255] (and 255 itself
// unless the table says otherwise) give an all-zero row.  Pure write-bound byte kernel: the output is
// walked as a flat array, 16 bytes per thread per store, the table comes from shared memory when it fits.
#include "common.cuh"

namespace mdseg {
namespace {

template <typename L, bool kSmem>
__global__ void __launch_bounds__(256) multihot_kernel(const L* __restrict__ labels, const uint8_t* __restrict__ table,
                                                       int C_uni, int64_t n_px, uint8_t* __restrict__ out) {
  extern __shared__ uint8_t s_table[];
  if (kSmem) {
    for (int i = threadIdx.x; i < 256 * C_uni; i += blockDim.x) s_table[i] = table[i];
    __syncthreads();
  }
  const uint8_t* tab = kSmem ? s_table : table;
  const int64_t total = n_px * C_uni;
  const int64_t n_vec = total / 16;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n_vec; v += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i0 = v * 16;
    int64_t p = i0 / C_uni;
    int u = (int)(i0 - p * C_uni);
    int lab = load_label<L>(labels, p);
    const uint8_t* row = ((unsigned)lab < 256u) ? tab + lab * C_uni : nullptr;
    uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const uint32_t b = row ? row[u] : 0u;
      w[k >> 2] |= b << (8 * (k & 3));
      if (++u == C_uni) {
        u = 0;
        ++p;
        if (p < n_px) {
          lab = load_label<L>(labels, p);
          row = ((unsigned)lab < 256u) ? tab + lab * C_uni : nullptr;
        }
      }
    }
    stg_stream_v4(out + i0, make_int4((int)w[0], (int)w[1], (int)w[2], (int)w[3]));
  }
  // ragged tail (< 16 bytes)
  for (int64_t i = n_vec * 16 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = i / C_uni;
    const int u = (int)(i - p * C_uni);
    const int lab = load_label<L>(labels, p);
    out[i] = ((unsigned)lab < 256u) ? tab[lab * C_uni + u] : (uint8_t)0;
  }
}

template <typename L>
int launch_multihot(const void* labels, const uint8_t* table, int C_uni, int64_t n_px, uint8_t* out, cudaStream_t s) {
  const size_t smem = (size_t)256 * C_uni;
  const bool use_smem = smem <= 100 * 1024;
  int64_t blocks = ceil_div64(ceil_div64(n_px * C_uni, 16), 256);
  const int64_t cap = (int64_t)sm_count() * (use_smem && smem > 48 * 1024 ? 2 : 8);
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  if (use_smem) {
    auto k = multihot_kernel<L, true>;
    if (smem > 48 * 1024) MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<(unsigned)blocks, 256, smem, s>>>((const L*)labels, table, C_uni, n_px, out);
  } else {
    multihot_kernel<L, false><<<(unsigned)blocks, 256, 0, s>>>((const L*)labels, table, C_uni, n_px, out);
  }
  MDSEG_LAUNCH_OK();
  return 0;
}

}  // namespace
}  // namespace mdseg

extern "C" int mdseg_multihot_remap(const void* labels, int label_dtype, const uint8_t* table, int C_uni, int64_t n_px,
                                    uint8_t* out, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(C_uni > 0 && C_uni <= 65535 && n_px >= 0, "mdseg_multihot_remap: bad shape");
  if (n_px == 0) return 0;
  MDSEG_REQUIRE(labels && table && out, "mdseg_multihot_remap: null pointer");
  MDSEG_REQUIRE(((uintptr_t)out & 15) == 0, "mdseg_multihot_remap: out must be 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  return with_int_type(label_dtype, "mdseg_multihot_remap", "label dtype", [&](auto l) {
    return launch_multihot<typename decltype(l)::type>(labels, table, C_uni, n_px, out, s);
  });
}
