// tma_util.cu — host side of tma_util.cuh: tensor-map construction and the fast-path geometry test.
#include "tma_util.cuh"

namespace mdseg {
namespace tma {

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}

int bind_primary_context() {
  static thread_local bool bound = false;
  if (!bound) {
    MDSEG_CUDA_OK(cudaFree(nullptr));
    bound = true;
  }
  return 0;
}

namespace {

// largest number of destinations that fall into one cell (cells fold the last source index, see axis_cell)
int max_cell_population(float scale, int n_in, int n_out) {
  int best = 0, run = 0, prev = -1;
  for (int dst = 0; dst < n_out; ++dst) {
    const float s = scale * (float)dst;
    int c = (int)s;
    if (c > n_in - 2) c = n_in - 2;
    if (c == prev) {
      ++run;
    } else {
      if (c < prev) return 1 << 30;  // not monotone: never on the fast path
      run = 1;
      prev = c;
    }
    best = run > best ? run : best;
  }
  return best;
}

}  // namespace

namespace {
// channel maximum of the low-res sources: cmax[b, y, x] = max_c src[b, c, y, x]
__global__ void __launch_bounds__(256)
channel_max_kernel(const mdseg_src_table src, const int32_t* __restrict__ dataset_ids, int64_t hw) {
  const int b = blockIdx.y;
  const int d = dataset_ids ? dataset_ids[b] : 0;
  if (d < 0 || d >= src.n_datasets) return;
  const float* img = (const float*)src.base[d] + (int64_t)b * src.image_stride[d];
  const int C = src.C[d];
  float* out = src.cmax + (int64_t)b * hw;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < hw / 4; q += (int64_t)gridDim.x * blockDim.x) {
    float4 m = *reinterpret_cast<const float4*>(img + q * 4);
    for (int c = 1; c < C; ++c) {
      const float4 v = *reinterpret_cast<const float4*>(img + (int64_t)c * hw + q * 4);
      m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
    }
    *reinterpret_cast<float4*>(out + q * 4) = m;
  }
}
}  // namespace

int channel_max(const mdseg_src_table& src, const int32_t* dataset_ids, int n_images, int64_t hw, cudaStream_t s) {
  int64_t bx = ceil_div64(hw / 4, 256);
  const int64_t want = ceil_div64((int64_t)sm_count() * 8, n_images);
  if (bx > want) bx = want;
  if (bx < 1) bx = 1;
  channel_max_kernel<<<dim3((unsigned)bx, (unsigned)n_images), 256, 0, s>>>(src, dataset_ids, hw);
  MDSEG_LAUNCH_OK();
  return 0;
}

bool fast_geometry(const mdseg_src_table& src, const Geom& gm) {
  if (src.dtype != MDSEG_F32) return false;
  if (gm.h < 2 || gm.w < 2 || gm.w % 4 != 0) return false;
  if (gm.H < gm.h || gm.W < gm.w) return false;  // up-sampling only
  if (gm.H > 5 * gm.h + 5 || gm.W > 5 * gm.w + 5) return false;
  if (max_cell_population(gm.ym.scale, gm.h, gm.H) > 5) return false;
  if (max_cell_population(gm.xm.scale, gm.w, gm.W) > 5) return false;
  for (int i = 0; i < src.n_datasets; ++i) {
    if (src.C[i] > 254) return false;  // labels are staged as bytes, 255 = "no gradient"
    if (((uintptr_t)src.base[i] & 15) != 0 || (src.image_stride[i] % 4) != 0) return false;
  }
  return encode_fn() != nullptr;
}

int make_maps(const mdseg_src_table& src, const Geom& gm, int n_images, int box_w, int box_h, int box_c, Maps* out) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available in this driver");
    return 1;
  }
  if (int rc = bind_primary_context()) return rc;
  for (int i = 0; i < src.n_datasets; ++i) {
    const int calloc = src.C_alloc[i] > 0 ? src.C_alloc[i] : src.C[i];
    cuuint64_t dims[4] = {(cuuint64_t)gm.w, (cuuint64_t)gm.h, (cuuint64_t)calloc, (cuuint64_t)n_images};
    cuuint64_t strides[3] = {(cuuint64_t)gm.w * 4, (cuuint64_t)gm.h * gm.w * 4, (cuuint64_t)src.image_stride[i] * 4};
    cuuint32_t box[4] = {(cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)box_c, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&out->m[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(src.base[i]), dims, strides, box,
                     estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("cuTensorMapEncodeTiled failed for dataset %d (CUresult %d)", i, (int)r);
      return 1;
    }
  }
  return 0;
}

}  // namespace tma
}  // namespace mdseg
