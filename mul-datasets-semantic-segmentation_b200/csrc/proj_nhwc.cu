// proj_nhwc.cu — the sparse bipartite projection and its adjoint for channels_last (NHWC) unified logits, and the
// layout moves of the aux heads' channels_last sources (DESIGN §3.12).
//
// A model run with memory_format=torch.channels_last hands the loss x[b, p, c] (pixel-major).  The NCHW kernels of
// proj.cu would need a full x.contiguous() copy first (3 GB read + 3 GB written at cfg3) and hand back an NCHW gradient
// that autograd converts again.  Here:
//  * forward: TP consecutive pixels x C_uni channels are one contiguous chunk of x; it arrives in shared memory with
//    one cp.async.bulk, lanes map to pixels and walk the CSR rows from there, so y (NCHW planes, what the fused
//    upsample + CE kernels read) is stored coalesced.  Each y[n, p] is the fmaf chain of proj_fwd_sparse_kernel in the
//    same CSR order: y and the channel maximum are bit-identical to mdseg_proj_fwd on x.contiguous().
//  * backward: the dy rows of a pixel tile are staged in shared memory and every thread produces consecutive elements
//    of the contiguous NHWC gradient tile (CSC walk per unified class, the order of proj_bwd_sparse_kernel), written
//    with 16-byte stores.
//  * aux heads: a gather-transpose packs the rows of each head's own images into one planar buffer in the source
//    dtype (what mdseg_up_ce_fwd reads), and a scatter-transpose writes the gradient rows back into every head's NHWC
//    gradient, zeros for the images of other datasets.
#include "tma_util.cuh"

namespace mdseg {
namespace {

constexpr int kThreads = 256;
constexpr int kTileBytesPerChannel = 128;  // TP * sizeof(T): 32 fp32 pixels or 64 16-bit pixels per tile
constexpr int kBwdTP = 64;                 // pixels per backward tile

// ---------------------------------------------------------------------------
// forward: one CTA = TP pixels of one image; warp w computes the dataset classes n = w, w + 8, ...
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads)
proj_fwd_nhwc_kernel(const T* __restrict__ x, const mdseg_graph_table tab, const int32_t* __restrict__ dataset_ids,
                     int64_t hw, float* __restrict__ y, int y_cmax, float* __restrict__ cmax, int* err_flag) {
  constexpr int TP = kTileBytesPerChannel / (int)sizeof(T);
  constexpr int PG = TP / 32;  // pixels per lane
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ float red[kThreads / 32][TP];
  const int b = blockIdx.y;
  const int d = dataset_ids ? dataset_ids[b] : 0;
  if (d < 0 || d >= tab.n_datasets) {
    if (threadIdx.x == 0 && blockIdx.x == 0 && err_flag) atomicOr(err_flag, MDSEG_ERR_DATASET_ID);
    return;
  }
  const mdseg_sparse_graph g = tab.g[d];
  const int Cu = tab.C_uni;
  const int64_t p0 = (int64_t)blockIdx.x * TP;
  const int np = (int)((hw - p0) < TP ? (hw - p0) : TP);
  const T* src = x + ((int64_t)b * hw + p0) * Cu;
  const uint32_t bytes = (uint32_t)np * Cu * sizeof(T);
  T* xs = reinterpret_cast<T*>(smem);
  if ((((uintptr_t)src | bytes) & 15) == 0) {
    if (threadIdx.x == 0) {
      tma::mbar_init(&bar, 1);
      tma::mbar_fence_init();
      tma::mbar_expect_tx(&bar, bytes);
      tma::bulk_g2s(xs, src, bytes, &bar);
    }
    __syncthreads();  // the barrier is initialised before anyone polls it
    tma::mbar_wait(&bar, 0);
  } else {  // odd C_uni * e, a storage offset or an unaligned image start: plain element copies into the same layout
    for (int e = threadIdx.x; e < np * Cu; e += kThreads) xs[e] = src[e];
    __syncthreads();
  }

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float mx[PG];
#pragma unroll
  for (int i = 0; i < PG; ++i) mx[i] = -3.402823466e38f;
  int px[PG];
#pragma unroll
  for (int i = 0; i < PG; ++i) px[i] = (i * 32 + lane < np ? i * 32 + lane : 0) * Cu;  // clamped reads stay in the tile
  float* yb = y + (int64_t)b * y_cmax * hw + p0;
  for (int n = warp; n < g.C_ds; n += kThreads / 32) {
    float acc[PG];
#pragma unroll
    for (int i = 0; i < PG; ++i) acc[i] = 0.f;
    const int j0 = __ldg(g.csr_ptr + n), j1 = __ldg(g.csr_ptr + n + 1);
    for (int j = j0; j < j1; ++j) {
      const int c = __ldg(g.csr_col + j);
      const float wv = g.csr_val ? __ldg(g.csr_val + j) : 1.f;
#pragma unroll
      for (int i = 0; i < PG; ++i) acc[i] = fmaf(wv, to_f32<T>(xs[px[i] + c]), acc[i]);
    }
#pragma unroll
    for (int i = 0; i < PG; ++i) {
      mx[i] = fmaxf(mx[i], acc[i]);
      if (i * 32 + lane < np) yb[(int64_t)n * hw + i * 32 + lane] = acc[i];
    }
  }
  if (cmax) {  // per-pixel channel maximum: fmaxf is order-free, so the warps' partial maxima combine to the same value
#pragma unroll
    for (int i = 0; i < PG; ++i) red[warp][i * 32 + lane] = mx[i];
    __syncthreads();
    for (int p = threadIdx.x; p < np; p += kThreads) {
      float m = red[0][p];
#pragma unroll
      for (int w = 1; w < kThreads / 32; ++w) m = fmaxf(m, red[w][p]);
      cmax[(int64_t)b * hw + p0 + p] = m;
    }
  }
}

// ---------------------------------------------------------------------------
// backward: dx[b, p, c] = Σ_{n in CSC column c} val * (dyA + dyB)[b, n, p], one CTA = kBwdTP pixels of one image.
// Thread t produces the V consecutive elements [V t, V t + V) of the contiguous NHWC tile (strided over the tile).
// ---------------------------------------------------------------------------
template <typename T, int V> __device__ __forceinline__ void store_run(T* p, const float (&v)[V], bool vec, int n_left) {
  if (vec && n_left >= V) {
    VecLoad<T, V>::store(p, v);
  } else {
#pragma unroll
    for (int i = 0; i < V; ++i)
      if (i < n_left) p[i] = from_f32<T>(v[i]);
  }
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
proj_bwd_nhwc_kernel(const float* __restrict__ dyA, const float* __restrict__ dyB, int y_cmax,
                     const mdseg_graph_table tab, const int32_t* __restrict__ dataset_ids, int64_t hw,
                     T* __restrict__ dx) {
  constexpr int V = 16 / (int)sizeof(T);
  constexpr int LD = kBwdTP + 1;  // row stride of the staged dy: lanes reading different classes of one pixel spread
  extern __shared__ __align__(16) float dys[];
  const int b = blockIdx.y;
  const int d = dataset_ids ? dataset_ids[b] : 0;
  const int Cu = tab.C_uni;
  const int64_t p0 = (int64_t)blockIdx.x * kBwdTP;
  const int np = (int)((hw - p0) < kBwdTP ? (hw - p0) : kBwdTP);
  const int n_el = np * Cu;
  T* out = dx + ((int64_t)b * hw + p0) * Cu;
  const bool vec = ((uintptr_t)out & 15) == 0;
  if (d < 0 || d >= tab.n_datasets) {  // image not part of the loss: zero gradient
    float z[V];
#pragma unroll
    for (int i = 0; i < V; ++i) z[i] = 0.f;
    for (int e = threadIdx.x * V; e < n_el; e += kThreads * V) store_run<T, V>(out + e, z, vec, n_el - e);
    return;
  }
  const mdseg_sparse_graph g = tab.g[d];
  // column-one-hot graphs: the one (class, value) of every unified class staged next to dy, one shared load per element
  int* col_n = reinterpret_cast<int*>(dys + (size_t)g.C_ds * LD);
  float* col_v = reinterpret_cast<float*>(col_n + Cu);
  if (g.col_onehot) {
    for (int c = threadIdx.x; c < Cu; c += kThreads) {
      const int j0 = __ldg(g.csc_ptr + c), j1 = __ldg(g.csc_ptr + c + 1);
      col_n[c] = j0 < j1 ? __ldg(g.csc_row + j0) * LD : -1;
      col_v[c] = j0 < j1 && g.csc_val ? __ldg(g.csc_val + j0) : 1.f;
    }
  }
  const float* ya = dyA + (int64_t)b * y_cmax * hw + p0;
  const float* yb = dyB ? dyB + (int64_t)b * y_cmax * hw + p0 : nullptr;
  for (int e = threadIdx.x; e < g.C_ds * kBwdTP; e += kThreads) {
    const int n = e / kBwdTP, p = e - n * kBwdTP;
    float v = 0.f;
    if (p < np) {
      v = ya[(int64_t)n * hw + p];
      if (yb) v += yb[(int64_t)n * hw + p];
    }
    dys[n * LD + p] = v;
  }
  __syncthreads();
  for (int e = threadIdx.x * V; e < n_el; e += kThreads * V) {
    int p = e / Cu, c = e - p * Cu;
    float o[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
      float acc = 0.f;
      if (g.col_onehot) {  // the row walk of proj_bwd_sparse_kernel: one product, zero for an unmapped class
        const int r = col_n[c];
        if (r >= 0) acc = col_v[c] * dys[r + p];
      } else {
        const int j0 = __ldg(g.csc_ptr + c), j1 = __ldg(g.csc_ptr + c + 1);
        for (int j = j0; j < j1; ++j)
          acc = fmaf(g.csc_val ? __ldg(g.csc_val + j) : 1.f, dys[__ldg(g.csc_row + j) * LD + p], acc);
      }
      o[i] = acc;
      if (++c == Cu) {  // the run crosses into the next pixel (past the tile end only for values never stored)
        c = 0;
        if (p + 1 < np) ++p;
      }
    }
    store_run<T, V>(out + e, o, vec, n_el - e);
  }
}

// ---------------------------------------------------------------------------
// aux heads: NHWC head sources <-> planar [n_images, C_alloc, h, w] rows of each image's own head.
// 32 pixels x 32 channels per CTA through a padded shared tile.  kToPlanar: image b's rows of head ids[b] are copied
// into the planar buffer.  Otherwise every head's NHWC gradient is written: the planar rows for the head of the image,
// zeros for the other heads.
// ---------------------------------------------------------------------------
template <typename T, bool kToPlanar>
__global__ void __launch_bounds__(kThreads)
nhwc_planar_kernel(const mdseg_src_table nhwc, const mdseg_src_table planar, const int32_t* __restrict__ dataset_ids,
                   int64_t hw) {
  __shared__ T t[32][33];
  const int b = blockIdx.z;
  const int own = dataset_ids ? dataset_ids[b] : 0;
  const int64_t p0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int d = 0; d < nhwc.n_datasets; ++d) {
    const int C = nhwc.C[d];
    if (c0 >= C) continue;
    if (kToPlanar && d != own) continue;
    T* hd = (T*)nhwc.base[d] + (int64_t)b * nhwc.image_stride[d];
    if (d != own) {  // gradient of a head for an image of another dataset
      for (int r = ty; r < 32; r += 8)
        if (p0 + r < hw && c0 + tx < C) hd[(p0 + r) * C + c0 + tx] = from_f32<T>(0.f);
      continue;
    }
    T* pl = (T*)planar.base[d] + (int64_t)b * planar.image_stride[d];
    if (kToPlanar) {
      for (int r = ty; r < 32; r += 8)
        if (p0 + r < hw && c0 + tx < C) t[r][tx] = hd[(p0 + r) * C + c0 + tx];
      __syncthreads();
      for (int r = ty; r < 32; r += 8)
        if (c0 + r < C && p0 + tx < hw) pl[(int64_t)(c0 + r) * hw + p0 + tx] = t[tx][r];
    } else {
      for (int r = ty; r < 32; r += 8)
        if (c0 + r < C && p0 + tx < hw) t[r][tx] = pl[(int64_t)(c0 + r) * hw + p0 + tx];
      __syncthreads();
      for (int r = ty; r < 32; r += 8)
        if (p0 + r < hw && c0 + tx < C) hd[(p0 + r) * C + c0 + tx] = t[tx][r];
    }
    __syncthreads();
  }
}

int check_sparse_table(const mdseg_graph_table* t, const char* who) {
  MDSEG_REQUIRE(graph_header_ok(t) && t->C_uni <= MDSEG_NHWC_MAX_CUNI,
                "%s: bad graph table (C_uni must be in [1, %d])", who, MDSEG_NHWC_MAX_CUNI);
  for (int i = 0; i < t->n_datasets; ++i) {
    const mdseg_sparse_graph& g = t->g[i];
    MDSEG_REQUIRE(g.C_ds > 0 && g.C_ds <= MDSEG_NHWC_MAX_CDS, "%s: dataset %d has C_ds outside [1, %d]", who, i,
                  MDSEG_NHWC_MAX_CDS);
    MDSEG_REQUIRE(!g.dense && g.csr_ptr && g.csc_ptr && (g.nnz == 0 || (g.csr_col && g.csc_row)),
                  "%s: dataset %d needs a sparse graph (dense graphs take the NCHW kernels)", who, i);
  }
  return 0;
}

template <typename T>
int launch_fwd(const void* x, const mdseg_graph_table* t, const int32_t* ids, int n_images, int64_t hw, float* y,
               int y_cmax, float* cmax, int32_t* ef, cudaStream_t s) {
  constexpr int TP = kTileBytesPerChannel / (int)sizeof(T);
  const size_t smem = (size_t)kTileBytesPerChannel * t->C_uni;
  auto k = proj_fwd_nhwc_kernel<T>;
  if (smem > 48 * 1024) MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((unsigned)ceil_div64(hw, TP), (unsigned)n_images);
  k<<<grid, kThreads, smem, s>>>((const T*)x, *t, ids, hw, y, y_cmax, cmax, ef);
  MDSEG_LAUNCH_OK();
  return 0;
}

template <typename T>
int launch_bwd(const float* dyA, const float* dyB, int y_cmax, const mdseg_graph_table* t, const int32_t* ids,
               int n_images, int64_t hw, void* dx, cudaStream_t s) {
  const size_t smem = (size_t)max_c_ds(t) * (kBwdTP + 1) * sizeof(float) + (size_t)t->C_uni * 8;
  auto k = proj_bwd_nhwc_kernel<T>;
  if (smem > 48 * 1024) MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((unsigned)ceil_div64(hw, kBwdTP), (unsigned)n_images);
  k<<<grid, kThreads, smem, s>>>(dyA, dyB, y_cmax, *t, ids, hw, (T*)dx);
  MDSEG_LAUNCH_OK();
  return 0;
}

template <bool kToPlanar>
int launch_move(const mdseg_src_table* nhwc, const mdseg_src_table* planar, const int32_t* ids, int n_images, int h,
                int w, cudaStream_t s, const char* who) {
  MDSEG_REQUIRE(src_count_ok(nhwc) && planar && planar->n_datasets == nhwc->n_datasets && planar->dtype == nhwc->dtype,
                "%s: bad source / destination table", who);
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0, "%s: bad shape", who);
  if (n_images == 0) return 0;
  const int64_t hw = (int64_t)h * w;
  int cm = 0;
  for (int i = 0; i < nhwc->n_datasets; ++i) {
    MDSEG_REQUIRE(nhwc->base[i] && planar->base[i] && nhwc->C[i] > 0 && planar->C[i] == nhwc->C[i] &&
                      nhwc->image_stride[i] >= hw * nhwc->C[i] && planar->image_stride[i] >= hw * nhwc->C[i],
                  "%s: head %d does not match", who, i);
    cm = nhwc->C[i] > cm ? nhwc->C[i] : cm;
  }
  MDSEG_REQUIRE(ceil_div64(hw, 32) <= 0x7fffffff, "%s: image too large", who);
  dim3 grid((unsigned)ceil_div64(hw, 32), (unsigned)((cm + 31) / 32), (unsigned)n_images);
  return with_float_type(nhwc->dtype, who, "dtype", [&](auto t) {
    nhwc_planar_kernel<typename decltype(t)::type, kToPlanar><<<grid, kThreads, 0, s>>>(*nhwc, *planar, ids, hw);
    MDSEG_LAUNCH_OK();
    return 0;
  });
}

}  // namespace
}  // namespace mdseg

extern "C" int mdseg_proj_fwd_nhwc(const void* x, int dtype, const mdseg_graph_table* graphs,
                                   const int32_t* dataset_ids, int n_images, int h, int w, float* y, int y_cmax,
                                   float* cmax_out, int32_t* err_flag, void* stream) {
  using namespace mdseg;
  if (int rc = check_sparse_table(graphs, "mdseg_proj_fwd_nhwc")) return rc;
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0, "mdseg_proj_fwd_nhwc: bad shape");
  MDSEG_REQUIRE(y_cmax >= max_c_ds(graphs), "mdseg_proj_fwd_nhwc: y_cmax %d < max C_ds %d", y_cmax, max_c_ds(graphs));
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(x && y, "mdseg_proj_fwd_nhwc: null pointer");
  const int64_t hw = (int64_t)h * w;
  cudaStream_t s = (cudaStream_t)stream;
  return with_float_type(dtype, "mdseg_proj_fwd_nhwc", "dtype", [&](auto t) {
    return launch_fwd<typename decltype(t)::type>(x, graphs, dataset_ids, n_images, hw, y, y_cmax, cmax_out, err_flag,
                                                  s);
  });
}

extern "C" int mdseg_proj_bwd_nhwc(const float* dyA, const float* dyB, int y_cmax, const mdseg_graph_table* graphs,
                                   const int32_t* dataset_ids, int n_images, int h, int w, void* dx, int dtype,
                                   void* stream) {
  using namespace mdseg;
  if (int rc = check_sparse_table(graphs, "mdseg_proj_bwd_nhwc")) return rc;
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0, "mdseg_proj_bwd_nhwc: bad shape");
  MDSEG_REQUIRE(y_cmax >= max_c_ds(graphs), "mdseg_proj_bwd_nhwc: y_cmax %d < max C_ds %d", y_cmax, max_c_ds(graphs));
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(dyA && dx, "mdseg_proj_bwd_nhwc: null pointer");
  const int64_t hw = (int64_t)h * w;
  cudaStream_t s = (cudaStream_t)stream;
  return with_float_type(dtype, "mdseg_proj_bwd_nhwc", "dtype", [&](auto t) {
    return launch_bwd<typename decltype(t)::type>(dyA, dyB, y_cmax, graphs, dataset_ids, n_images, hw, dx, s);
  });
}

extern "C" int mdseg_nhwc_to_planar(const mdseg_src_table* nhwc, const int32_t* dataset_ids, int n_images, int h, int w,
                                    const mdseg_src_table* planar, void* stream) {
  return mdseg::launch_move<true>(nhwc, planar, dataset_ids, n_images, h, w, (cudaStream_t)stream,
                                  "mdseg_nhwc_to_planar");
}

extern "C" int mdseg_planar_to_nhwc(const mdseg_src_table* planar, const int32_t* dataset_ids, int n_images, int h,
                                    int w, const mdseg_src_table* nhwc, void* stream) {
  return mdseg::launch_move<false>(nhwc, planar, dataset_ids, n_images, h, w, (cudaStream_t)stream,
                                   "mdseg_planar_to_nhwc");
}
