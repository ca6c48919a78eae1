// proj.cu — bipartite unified->dataset logit projection and its adjoints
// (SURVEY §8 row a5 and the projection part of a9).
//
// Reference work replaced (lib/loss/loss_cross_datasets.py:1006, :997/:1000 for
// the soft/max pair, lib/models/semseg.py:344, lib/models/HRNetv2.py:655):
//   remap_logit = torch.einsum('bchw, nc -> bnhw', logits[dataset_ids==i], bi_graphs[i])
// ATen: bool-mask gather of the image rows + permute/contiguous + cuBLAS bmm per
// dataset.  Here one launch covers every image of every dataset; each image
// looks up its dataset's graph from a by-value table, so ids may come in any
// order (MultiSetReader batches, lib/MultiSetReader.py:26-34).
//
// Two regimes, chosen per dataset by the graph descriptor:
//  * sparse (SEG stage: 0/1 column-one-hot graphs from UOT / pretrain, and the
//    general 0/1 ClassRemap matrix): CSR walk, y[n] = Σ_{c in row n} v*x[c].
//    Each unified channel plane is read once with 128-bit loads; exact when the
//    values are 0/1.  HBM bound: (C_uni*e + C_ds*4)/16 bytes per label pixel.
//  * dense (GNN stage, graphs with grad): shared-memory tiled FFMA contraction
//    (fp32 exact accumulate; the tensor-core variant is a later round, see
//    DESIGN.md).
#include "common.cuh"

namespace mdseg {
namespace {

// ---------------------------------------------------------------------------
// sparse forward: thread = PX consecutive low-res pixels of one image
// ---------------------------------------------------------------------------
template <typename T, int PX>
__global__ void __launch_bounds__(256)
proj_fwd_sparse_kernel(const T* __restrict__ x, const mdseg_graph_table tab, const int32_t* __restrict__ dataset_ids,
                       int64_t hw, float* __restrict__ y, int y_cmax, float* __restrict__ cmax, int* err_flag) {
  const int b = blockIdx.y;
  const int d = dataset_ids ? dataset_ids[b] : 0;
  if (d < 0 || d >= tab.n_datasets) {
    if (threadIdx.x == 0 && blockIdx.x == 0 && err_flag) atomicOr(err_flag, MDSEG_ERR_DATASET_ID);
    return;
  }
  const mdseg_sparse_graph g = tab.g[d];
  if (g.dense) return;  // handled by the dense kernel
  const T* xb = x + (int64_t)b * tab.C_uni * hw;
  float* yb = y + (int64_t)b * y_cmax * hw;
  const int64_t n_groups = hw / PX;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n_groups; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = q * PX;
    float mx[PX];
#pragma unroll
    for (int i = 0; i < PX; ++i) mx[i] = -3.402823466e38f;
    for (int n = 0; n < g.C_ds; ++n) {
      float acc[PX];
#pragma unroll
      for (int i = 0; i < PX; ++i) acc[i] = 0.f;
      const int j0 = __ldg(g.csr_ptr + n), j1 = __ldg(g.csr_ptr + n + 1);
      // up to 8 planes of a class in flight at once (predicated), accumulated in CSR order: a class of the 7-dataset
      // graphs has 5.9 unified channels on average, so most classes cost one memory round trip instead of 1 + (n mod 4)
      // (the loads stay in their 16-byte raw form until they are accumulated: widening eight bf16 planes to fp32 up
      // front costs 64 registers and most of the occupancy)
      for (int j = j0; j < j1; j += 8) {
        typename VecLoad<T, PX>::Raw raw[8];
        float wv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (j + u < j1) {
            const int c = __ldg(g.csr_col + j + u);
            wv[u] = g.csr_val ? __ldg(g.csr_val + j + u) : 1.f;
            raw[u] = VecLoad<T, PX>::raw(xb + (int64_t)c * hw + p);
          }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (j + u < j1) {
            float v[PX];
            VecLoad<T, PX>::unpack(raw[u], v);
#pragma unroll
            for (int i = 0; i < PX; ++i) acc[i] = fmaf(wv[u], v[i], acc[i]);
          }
        }
      }
      float* dst = yb + (int64_t)n * hw + p;
#pragma unroll
      for (int i = 0; i < PX; ++i) mx[i] = fmaxf(mx[i], acc[i]);
      if constexpr (PX == 1) {
        dst[0] = acc[0];
      } else {
#pragma unroll
        for (int i = 0; i < PX; i += 4)
          *reinterpret_cast<float4*>(dst + i) = make_float4(acc[i], acc[i + 1], acc[i + 2], acc[i + 3]);
      }
    }
    if (cmax) {  // per-pixel channel maximum, the softmax shift of the fused upsample+CE kernels
#pragma unroll
      for (int i = 0; i < PX; ++i) cmax[(int64_t)b * hw + p + i] = mx[i];
    }
  }
}

// ---------------------------------------------------------------------------
// sparse backward: dx[c] = Σ_n G[n,c] (dyA[n] + dyB[n])
// column-one-hot graphs walk the rows (each dy plane read once, each dx plane
// written once); general sparse graphs walk the columns.
// ---------------------------------------------------------------------------
template <int PX> __device__ __forceinline__ void load_dy(const float* a, const float* b, float (&o)[PX]) {
  if constexpr (PX == 1) {
    o[0] = a[0] + (b ? b[0] : 0.f);
  } else {
#pragma unroll
    for (int i = 0; i < PX; i += 4) {
      float4 u = *reinterpret_cast<const float4*>(a + i);
      if (b) {
        float4 w = *reinterpret_cast<const float4*>(b + i);
        u.x += w.x; u.y += w.y; u.z += w.z; u.w += w.w;
      }
      o[i] = u.x; o[i + 1] = u.y; o[i + 2] = u.z; o[i + 3] = u.w;
    }
  }
}

template <typename T, int PX>
__global__ void __launch_bounds__(256)
proj_bwd_sparse_kernel(const float* __restrict__ dyA, const float* __restrict__ dyB, int y_cmax,
                       const mdseg_graph_table tab, const int32_t* __restrict__ dataset_ids, int64_t hw,
                       T* __restrict__ dx) {
  const int b = blockIdx.y;
  const int d = dataset_ids ? dataset_ids[b] : 0;
  T* dxb = dx + (int64_t)b * tab.C_uni * hw;
  const int64_t n_groups = hw / PX;
  float zero[PX];
#pragma unroll
  for (int i = 0; i < PX; ++i) zero[i] = 0.f;
  if (d < 0 || d >= tab.n_datasets) {  // image not part of the loss: zero gradient
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n_groups; q += (int64_t)gridDim.x * blockDim.x)
      for (int c = 0; c < tab.C_uni; ++c) VecLoad<T, PX>::store(dxb + (int64_t)c * hw + q * PX, zero);
    return;
  }
  const mdseg_sparse_graph g = tab.g[d];
  if (g.dense) return;
  const float* ya = dyA + (int64_t)b * y_cmax * hw;
  const float* yb = dyB ? dyB + (int64_t)b * y_cmax * hw : nullptr;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n_groups; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = q * PX;
    if (g.col_onehot) {
      for (int n = 0; n < g.C_ds; ++n) {
        float gy[PX];
        load_dy<PX>(ya + (int64_t)n * hw + p, yb ? yb + (int64_t)n * hw + p : nullptr, gy);
        const int j0 = __ldg(g.csr_ptr + n), j1 = __ldg(g.csr_ptr + n + 1);
        for (int j = j0; j < j1; ++j) {
          const int c = __ldg(g.csr_col + j);
          const float wv = g.csr_val ? __ldg(g.csr_val + j) : 1.f;
          float o[PX];
#pragma unroll
          for (int i = 0; i < PX; ++i) o[i] = wv * gy[i];
          VecLoad<T, PX>::store(dxb + (int64_t)c * hw + p, o);
        }
      }
      for (int c = 0; c < tab.C_uni; ++c)  // unmapped unified classes get a zero gradient
        if (__ldg(g.csc_ptr + c) == __ldg(g.csc_ptr + c + 1)) VecLoad<T, PX>::store(dxb + (int64_t)c * hw + p, zero);
    } else {
      for (int c = 0; c < tab.C_uni; ++c) {
        float acc[PX];
#pragma unroll
        for (int i = 0; i < PX; ++i) acc[i] = 0.f;
        const int j0 = __ldg(g.csc_ptr + c), j1 = __ldg(g.csc_ptr + c + 1);
        for (int j = j0; j < j1; ++j) {
          const int n = __ldg(g.csc_row + j);
          const float wv = g.csc_val ? __ldg(g.csc_val + j) : 1.f;
          float gy[PX];
          load_dy<PX>(ya + (int64_t)n * hw + p, yb ? yb + (int64_t)n * hw + p : nullptr, gy);
#pragma unroll
          for (int i = 0; i < PX; ++i) acc[i] = fmaf(wv, gy[i], acc[i]);
        }
        VecLoad<T, PX>::store(dxb + (int64_t)c * hw + p, acc);
      }
    }
  }
}

// ---------------------------------------------------------------------------
// dense contraction  out[o][p] = Σ_k Wt(o,k) * in[k][p]   (per image)
//   forward : o = dataset class n, k = unified class c, Wt(o,k) = G[n][c]
//   backward: o = unified class c, k = dataset class n, Wt(o,k) = G[n][c]
// CTA tile: 128 pixels x 32 outputs, K chunk 16, 256 threads, 4x4 outputs each.
// ---------------------------------------------------------------------------
constexpr int kTP = 128, kTO = 32, kTK = 16;

template <typename TIn, typename TOut, bool kFwd>
__global__ void __launch_bounds__(256)
proj_dense_kernel(const TIn* __restrict__ in, const float* __restrict__ in2, const mdseg_graph_table tab,
                  const int32_t* __restrict__ dataset_ids, int64_t hw, int in_cstride, int out_cstride,
                  TOut* __restrict__ out, unsigned skip_mask) {
  const int b = blockIdx.z;
  const int d = dataset_ids ? dataset_ids[b] : 0;
  if (d < 0 || d >= tab.n_datasets || ((skip_mask >> d) & 1u)) return;
  const mdseg_sparse_graph g = tab.g[d];
  if (!g.dense) return;
  const int K = kFwd ? tab.C_uni : g.C_ds;
  const int O = kFwd ? g.C_ds : tab.C_uni;
  const int o0 = blockIdx.y * kTO;
  if (o0 >= O) return;
  const int64_t p0 = (int64_t)blockIdx.x * kTP;

  __shared__ float Xs[kTK][kTP];
  __shared__ float Ws[kTK][kTO + 4];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const TIn* inb = in + (int64_t)b * in_cstride * hw;
  const float* in2b = in2 ? in2 + (int64_t)b * in_cstride * hw : nullptr;
  for (int k0 = 0; k0 < K; k0 += kTK) {
    // stage the input tile [16][128]
    for (int e = threadIdx.x; e < kTK * kTP; e += 256) {
      const int kk = e / kTP, pp = e % kTP;
      float v = 0.f;
      if (k0 + kk < K && p0 + pp < hw) {
        const int64_t idx = (int64_t)(k0 + kk) * hw + p0 + pp;
        v = to_f32<TIn>(inb[idx]);
        if (in2b) v += in2b[idx];
      }
      Xs[kk][pp] = v;
    }
    // stage the weight tile [16][32]
    for (int e = threadIdx.x; e < kTK * kTO; e += 256) {
      const int kk = e / kTO, oo = e % kTO;
      float v = 0.f;
      if (k0 + kk < K && o0 + oo < O)
        v = kFwd ? g.dense[(int64_t)(o0 + oo) * tab.C_uni + (k0 + kk)] : g.dense[(int64_t)(k0 + kk) * tab.C_uni + (o0 + oo)];
      Ws[kk][oo] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kTK; ++kk) {
      const float4 xv = *reinterpret_cast<const float4*>(&Xs[kk][tx * 4]);
      const float4 wv = *reinterpret_cast<const float4*>(&Ws[kk][ty * 4]);
      const float xa[4] = {xv.x, xv.y, xv.z, xv.w};
      const float wa[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(wa[i], xa[j], acc[i][j]);
    }
    __syncthreads();
  }
  TOut* outb = out + (int64_t)b * out_cstride * hw;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int o = o0 + ty * 4 + i;
    if (o >= O) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t p = p0 + tx * 4 + j;
      if (p < hw) outb[(int64_t)o * hw + p] = from_f32<TOut>(acc[i][j]);
    }
  }
}

// ---------------------------------------------------------------------------
// d bi_graph:  dG[n][c] += Σ_p (dyA+dyB)[n][p] * x[c][p]   (split over pixel slabs)
// CTA tile 32 n x 32 c, 256 threads (2x2 outputs each), pixel chunk 32.
// ---------------------------------------------------------------------------
constexpr int kGP = 32;

template <typename T>
__global__ void __launch_bounds__(256)
proj_dgraph_kernel(const T* __restrict__ x, const float* __restrict__ dyA, const float* __restrict__ dyB, int y_cmax,
                   const mdseg_graph_table tab, const int32_t* __restrict__ dataset_ids, int64_t hw, int64_t slab,
                   float* __restrict__ dG, long long dg_stride, unsigned skip_mask) {
  const int n_slabs = (int)((hw + slab - 1) / slab);
  const int b = blockIdx.z / n_slabs, sl = blockIdx.z % n_slabs;
  const int d = dataset_ids ? dataset_ids[b] : 0;
  if (d < 0 || d >= tab.n_datasets || ((skip_mask >> d) & 1u)) return;
  const mdseg_sparse_graph g = tab.g[d];
  const int n0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  if (n0 >= g.C_ds || c0 >= tab.C_uni) return;
  __shared__ float Ys[32][kGP + 1];
  __shared__ float Xs[32][kGP + 1];
  const int tn = threadIdx.x >> 4, tc = threadIdx.x & 15;  // 16 x 16 threads
  float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
  const T* xb = x + (int64_t)b * tab.C_uni * hw;
  const float* ya = dyA + (int64_t)b * y_cmax * hw;
  const float* yb = dyB ? dyB + (int64_t)b * y_cmax * hw : nullptr;
  const int64_t pbeg = (int64_t)sl * slab;
  const int64_t pend = (pbeg + slab < hw) ? pbeg + slab : hw;
  for (int64_t p0 = pbeg; p0 < pend; p0 += kGP) {
    for (int e = threadIdx.x; e < 32 * kGP; e += 256) {
      const int r = e / kGP, pp = e % kGP;
      const int64_t p = p0 + pp;
      float yv = 0.f, xv = 0.f;
      if (p < pend) {
        if (n0 + r < g.C_ds) {
          yv = ya[(int64_t)(n0 + r) * hw + p];
          if (yb) yv += yb[(int64_t)(n0 + r) * hw + p];
        }
        if (c0 + r < tab.C_uni) xv = to_f32<T>(xb[(int64_t)(c0 + r) * hw + p]);
      }
      Ys[r][pp] = yv;
      Xs[r][pp] = xv;
    }
    __syncthreads();
#pragma unroll
    for (int pp = 0; pp < kGP; ++pp) {
      const float y0 = Ys[tn * 2][pp], y1 = Ys[tn * 2 + 1][pp];
      const float x0 = Xs[tc * 2][pp], x1 = Xs[tc * 2 + 1][pp];
      acc[0][0] = fmaf(y0, x0, acc[0][0]); acc[0][1] = fmaf(y0, x1, acc[0][1]);
      acc[1][0] = fmaf(y1, x0, acc[1][0]); acc[1][1] = fmaf(y1, x1, acc[1][1]);
    }
    __syncthreads();
  }
  float* dg = dG + (long long)d * dg_stride;
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int n = n0 + tn * 2 + i, c = c0 + tc * 2 + j;
      if (n < g.C_ds && c < tab.C_uni && acc[i][j] != 0.f) atomicAdd(dg + (int64_t)n * tab.C_uni + c, acc[i][j]);
    }
}

bool any_dense(const mdseg_graph_table* t, unsigned skip_mask = 0) {
  for (int i = 0; i < t->n_datasets; ++i)
    if (t->g[i].dense && !((skip_mask >> i) & 1u)) return true;
  return false;
}
bool any_sparse(const mdseg_graph_table* t) {
  for (int i = 0; i < t->n_datasets; ++i)
    if (!t->g[i].dense) return true;
  return false;
}
int check_table(const mdseg_graph_table* t, const char* who) {
  MDSEG_REQUIRE(graph_header_ok(t), "%s: bad graph table", who);
  for (int i = 0; i < t->n_datasets; ++i) {
    const mdseg_sparse_graph& g = t->g[i];
    MDSEG_REQUIRE(g.C_ds > 0, "%s: dataset %d has C_ds <= 0", who, i);
    MDSEG_REQUIRE(g.dense || (g.csr_ptr && g.csc_ptr && (g.nnz == 0 || (g.csr_col && g.csc_row))),
                  "%s: dataset %d has neither a dense nor a sparse graph", who, i);
  }
  return 0;
}

template <typename T>
int launch_fwd(const void* x, const mdseg_graph_table* t, const int32_t* ids, int n_images, int64_t hw, float* y,
               int y_cmax, float* cmax, int32_t* ef, unsigned skip_mask, cudaStream_t s) {
  constexpr int PXV = 16 / sizeof(T);
  if (any_sparse(t)) {
    const bool vec = (hw % PXV == 0) && ((((uintptr_t)x | (uintptr_t)y) & 15) == 0);
    const int64_t groups = vec ? hw / PXV : hw;
    int64_t bx = ceil_div64(groups, 256);
    int64_t want = ceil_div64((int64_t)sm_count() * 8, n_images);
    if (bx > want) bx = want;
    dim3 grid((unsigned)bx, (unsigned)n_images);
    if (vec) proj_fwd_sparse_kernel<T, PXV><<<grid, 256, 0, s>>>((const T*)x, *t, ids, hw, y, y_cmax, cmax, ef);
    else proj_fwd_sparse_kernel<T, 1><<<grid, 256, 0, s>>>((const T*)x, *t, ids, hw, y, y_cmax, cmax, ef);
    MDSEG_LAUNCH_OK();
  }
  if (any_dense(t, skip_mask)) {
    dim3 grid((unsigned)ceil_div64(hw, kTP), (unsigned)((max_c_ds(t) + kTO - 1) / kTO), (unsigned)n_images);
    proj_dense_kernel<T, float, true><<<grid, 256, 0, s>>>((const T*)x, nullptr, *t, ids, hw, t->C_uni, y_cmax, y,
                                                           skip_mask);
    MDSEG_LAUNCH_OK();
  }
  return 0;
}

template <typename T>
int launch_bwd(const float* dyA, const float* dyB, int y_cmax, const mdseg_graph_table* t, const int32_t* ids,
               int n_images, int64_t hw, void* dx, unsigned skip_mask, cudaStream_t s) {
  constexpr int PXV = 16 / sizeof(T);
  {  // the sparse kernel also zero-fills images with an invalid dataset id
    const bool vec = (hw % PXV == 0) && ((((uintptr_t)dx | (uintptr_t)dyA | (uintptr_t)dyB) & 15) == 0);
    const int64_t groups = vec ? hw / PXV : hw;
    int64_t bx = ceil_div64(groups, 256);
    int64_t want = ceil_div64((int64_t)sm_count() * 8, n_images);
    if (bx > want) bx = want;
    dim3 grid((unsigned)bx, (unsigned)n_images);
    if (vec) proj_bwd_sparse_kernel<T, PXV><<<grid, 256, 0, s>>>(dyA, dyB, y_cmax, *t, ids, hw, (T*)dx);
    else proj_bwd_sparse_kernel<T, 1><<<grid, 256, 0, s>>>(dyA, dyB, y_cmax, *t, ids, hw, (T*)dx);
    MDSEG_LAUNCH_OK();
  }
  if (any_dense(t, skip_mask)) {
    dim3 grid((unsigned)ceil_div64(hw, kTP), (unsigned)((t->C_uni + kTO - 1) / kTO), (unsigned)n_images);
    proj_dense_kernel<float, T, false><<<grid, 256, 0, s>>>(dyA, dyB, *t, ids, hw, y_cmax, t->C_uni, (T*)dx, skip_mask);
    MDSEG_LAUNCH_OK();
  }
  return 0;
}

template <typename T>
int launch_dgraph(const void* x, const float* dyA, const float* dyB, int y_cmax, const mdseg_graph_table* t,
                  const int32_t* ids, int n_images, int64_t hw, float* dG, long long dg_stride, unsigned skip_mask,
                  cudaStream_t s) {
  // pixel slabs: enough CTAs to fill the chip, at least 2048 px each
  int64_t slab = 2048;
  const int n_slabs = (int)ceil_div64(hw, slab);
  dim3 grid((unsigned)((t->C_uni + 31) / 32), (unsigned)((max_c_ds(t) + 31) / 32), (unsigned)(n_images * n_slabs));
  proj_dgraph_kernel<T><<<grid, 256, 0, s>>>((const T*)x, dyA, dyB, y_cmax, *t, ids, hw, slab, dG, dg_stride,
                                             skip_mask);
  MDSEG_LAUNCH_OK();
  return 0;
}

}  // namespace
}  // namespace mdseg

namespace mdseg {
// Projection of every dataset whose bit is clear in skip_mask (the tensor-core kernel of proj_tc.cu takes the rest).
int proj_fwd_rest(const void* x, int dtype, const mdseg_graph_table* graphs, const int32_t* dataset_ids, int n_images,
                  int h, int w, float* y, int y_cmax, float* cmax_out, int32_t* err_flag, unsigned skip_mask,
                  cudaStream_t s) {
  if (int rc = check_table(graphs, "mdseg_proj_fwd")) return rc;
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0, "mdseg_proj_fwd: bad shape");
  MDSEG_REQUIRE(y_cmax >= max_c_ds(graphs), "mdseg_proj_fwd: y_cmax %d < max C_ds %d", y_cmax, max_c_ds(graphs));
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(x && y, "mdseg_proj_fwd: null pointer");
  const int64_t hw = (int64_t)h * w;
  return with_float_type(dtype, "mdseg_proj_fwd", "dtype", [&](auto t) {
    return launch_fwd<typename decltype(t)::type>(x, graphs, dataset_ids, n_images, hw, y, y_cmax, cmax_out, err_flag,
                                                  skip_mask, s);
  });
}
}  // namespace mdseg

extern "C" int mdseg_proj_fwd(const void* x, int dtype, const mdseg_graph_table* graphs, const int32_t* dataset_ids,
                              int n_images, int h, int w, float* y, int y_cmax, float* cmax_out, int32_t* err_flag,
                              void* stream) {
  return mdseg::proj_fwd_rest(x, dtype, graphs, dataset_ids, n_images, h, w, y, y_cmax, cmax_out, err_flag, 0u,
                              (cudaStream_t)stream);
}

namespace mdseg {
// Adjoint of every dataset whose bit is clear in skip_mask (plus the zero fill of images without a dataset).
int proj_bwd_rest(const float* dyA, const float* dyB, int y_cmax, const mdseg_graph_table* graphs,
                  const int32_t* dataset_ids, int n_images, int h, int w, void* dx, int dtype, unsigned skip_mask,
                  cudaStream_t s) {
  if (int rc = check_table(graphs, "mdseg_proj_bwd")) return rc;
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0, "mdseg_proj_bwd: bad shape");
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(dyA && dx, "mdseg_proj_bwd: null pointer");
  const int64_t hw = (int64_t)h * w;
  return with_float_type(dtype, "mdseg_proj_bwd", "dtype", [&](auto t) {
    return launch_bwd<typename decltype(t)::type>(dyA, dyB, y_cmax, graphs, dataset_ids, n_images, hw, dx, skip_mask,
                                                  s);
  });
}
}  // namespace mdseg

extern "C" int mdseg_proj_bwd(const float* dyA, const float* dyB, int y_cmax, const mdseg_graph_table* graphs,
                              const int32_t* dataset_ids, int n_images, int h, int w, void* dx, int dtype,
                              void* stream) {
  return mdseg::proj_bwd_rest(dyA, dyB, y_cmax, graphs, dataset_ids, n_images, h, w, dx, dtype, 0u, (cudaStream_t)stream);
}

namespace mdseg {
// d bi_graph of every dataset whose bit is clear in skip_mask (atomic accumulation into dG).
int proj_dgraph_rest(const void* x, int dtype, const float* dyA, const float* dyB, int y_cmax,
                     const mdseg_graph_table* graphs, const int32_t* dataset_ids, int n_images, int h, int w, float* dG,
                     long long dg_stride, unsigned skip_mask, cudaStream_t s) {
  if (int rc = check_table(graphs, "mdseg_proj_bwd_graph")) return rc;
  MDSEG_REQUIRE(n_images >= 0 && h > 0 && w > 0, "mdseg_proj_bwd_graph: bad shape");
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(x && dyA && dG, "mdseg_proj_bwd_graph: null pointer");
  const int64_t hw = (int64_t)h * w;
  MDSEG_REQUIRE((int64_t)n_images * ceil_div64(hw, 2048) <= 65535, "mdseg_proj_bwd_graph: grid too large");
  bool any = false;
  for (int i = 0; i < graphs->n_datasets; ++i) any = any || !((skip_mask >> i) & 1u);
  if (!any) return 0;
  return with_float_type(dtype, "mdseg_proj_bwd_graph", "dtype", [&](auto t) {
    return launch_dgraph<typename decltype(t)::type>(x, dyA, dyB, y_cmax, graphs, dataset_ids, n_images, hw, dG,
                                                     dg_stride, skip_mask, s);
  });
}
}  // namespace mdseg

extern "C" int mdseg_proj_bwd_graph(const void* x, int dtype, const float* dyA, const float* dyB, int y_cmax,
                                    const mdseg_graph_table* graphs, const int32_t* dataset_ids, int n_images, int h,
                                    int w, float* dG, long long dg_stride, void* stream) {
  return mdseg::proj_dgraph_rest(x, dtype, dyA, dyB, y_cmax, graphs, dataset_ids, n_images, h, w, dG, dg_stride, 0u,
                                 (cudaStream_t)stream);
}
