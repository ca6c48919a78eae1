// proj_tc.cu — dense bipartite projection on the 5th-generation tensor cores (SURVEY §8 row a5, GNN stage).
//
// Reference work replaced (lib/loss/loss_cross_datasets.py:1006, :997/:1000; lib/models/semseg.py:344):
//   remap_logit = torch.einsum('bchw, nc -> bnhw', logits[dataset_ids==i], bi_graphs[i])
// with a DENSE fp32 bi_graph (soft adjacency of the GNN stage, requires_grad): a real
// [B_i*h*w, C_uni] x [C_uni, C_ds] contraction (cfg3 / ADE: 2*358*150 FLOP per low-res pixel).
//
// GEMM shape per CTA tile:  D[M = 128 pixels, N = C_ds padded to 16] += A[M, K] * B[N, K]^T,  K = C_uni.
//   * A = x^T: pixels are contiguous in HBM (NCHW), so a thread owns one pixel and half of a 32-channel
//     K-chunk (256 threads per 128-pixel tile), reads its 16 channels with warp-coalesced loads, converts
//     to 16-bit terms and writes them K-major into the canonical no-swizzle core-matrix layout (8 rows x
//     16 bytes per core matrix) in shared memory.
//   * B = G_d: split / converted ONCE by a prep kernel into the same layout in a caller-owned workspace;
//     each K-chunk arrives with one cp.async.bulk (mbarrier complete_tx).
//   * one elected thread issues tcgen05.mma (kind::f16, fp32 accumulate in TMEM); tcgen05.commit frees a
//     shared-memory stage and, after the last chunk, hands the accumulator to the epilogue;
//   * epilogue: tcgen05.ld (32 lanes x 32 bit, 16 columns at a time) -> coalesced fp32 stores of y[n][p].
// Precision: fp32 inputs are split into three bf16 terms each (x = xh + xm + xl, G likewise) and the six
// products of weight >= 2^-16 are accumulated (relative error ~2^-21, inside the 1e-5 parity bar without
// giving up fp32's range); bf16 / fp16 inputs take ONE product in their own type, G rounded to it — what
// autocast does to the reference einsum.
#include <type_traits>

#include "tma_util.cuh"

namespace mdseg {
// proj.cu: the same projection without the tensor-core datasets (bit d of skip_mask = dataset d is handled here)
int proj_fwd_rest(const void* x, int dtype, const mdseg_graph_table* graphs, const int32_t* dataset_ids, int n_images,
                  int h, int w, float* y, int y_cmax, float* cmax_out, int32_t* err_flag, unsigned skip_mask,
                  cudaStream_t s);

namespace {

using namespace tma;

constexpr int kTM = 128;      // pixels per tile = UMMA M
constexpr int kKB = 32;       // channels per shared-memory stage (two K = 16 MMA steps)
constexpr int kStagesTc = 2;
constexpr int kTcThreads = 2 * kTM;  // two threads per pixel: 16 channels of a chunk each
constexpr int kMaxN = 256;    // UMMA N limit

__host__ __device__ inline int pad16(int n) { return (n + 15) & ~15; }

struct TcArgs {
  const void* x;
  float* y;
  const int32_t* dataset_ids;
  const unsigned char* gw;               // prepared graphs (workspace)
  long long g_off[MDSEG_MAX_DATASETS];   // byte offset of dataset d's chunks
  int C_ds[MDSEG_MAX_DATASETS];
  unsigned tc_mask;                      // datasets handled by this kernel
  int n_datasets, C_uni, y_cmax;
  long long hw;
  int n_chunks;
  int a_stage_bytes, b_stage_bytes;      // per stage, all terms
  int fmt;                               // UMMA 16-bit format: 0 = F16, 1 = BF16
  // adjoint (dx = G^T (dyA + dyB)): K = C_ds, N = a tile of `nt` unified channels (blockIdx.z)
  const float* dyA;
  const float* dyB;                      // may be NULL
  void* dx;
  int nt;                                // unified channels per N tile, multiple of 16
  // forward N tiling (blockIdx.z): dataset d's classes in n_tiles_f[d] tiles of nt_f[d] rows (multiple of 16, <= 256);
  // one tile when C_ds <= 256 (the bipartite graphs), two or more for the prototype head (C_uni 358 classes)
  int nt_f[MDSEG_MAX_DATASETS];
  int n_tiles_f[MDSEG_MAX_DATASETS];
};

// 16 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld16_f32(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  tmem_ld16(taddr, r);
  tmem_wait_ld();
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Operands are K-major without swizzle (umma_desc kNoSwizzle): a core matrix is 8 rows x 16 bytes stored contiguously,
// `sbo` steps between 8-row groups (M / N direction), `lbo` between the core matrices adjacent in K.
// Instruction descriptor (cute::UMMA::InstrDescriptor): fp32 accumulate, A and B K-major, M = 128
__device__ __forceinline__ uint32_t umma_idesc(int fmt, int n) {
  return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTM >> 4) << 24);
}

// ---- 16-bit terms of fp32 values ------------------------------------------------------------------------
template <int TERMS> struct Split;  // pack two consecutive-K values into one 32-bit word per term
template <> struct Split<3> {
  static __device__ __forceinline__ void pair(float a, float b, int /*fmt*/, uint32_t (&o)[3]) {
    float ra = a, rb = b;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(ra, rb);
      o[t] = *reinterpret_cast<const uint32_t*>(&h);
      ra -= __low2float(h);
      rb -= __high2float(h);
    }
  }
};
template <> struct Split<1> {
  static __device__ __forceinline__ void pair(float a, float b, int fmt, uint32_t (&o)[1]) {
    if (fmt == 1) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
      o[0] = *reinterpret_cast<const uint32_t*>(&h);
    } else {
      const __half2 h = __floats2half2_rn(a, b);
      o[0] = *reinterpret_cast<const uint32_t*>(&h);
    }
  }
};

// ---- prep: G_d [C_ds, C_uni] fp32 -> per N tile, per K-chunk, per term, canonical K-major core-matrix layout ---------
// chunk (d, z, kc) holds TERMS blocks of [nt rows][32 k]: byte offset of (term t, row r, k) inside the chunk =
// t * nt * 64 + (k / 8) * (nt * 16) + r * 16 + (k % 8) * 2; row r of tile z is class z * nt + r.
template <int TERMS>
__global__ void __launch_bounds__(256) proj_tc_prep_kernel(const mdseg_graph_table tab, unsigned tc_mask, int n_chunks,
                                                           int fmt, unsigned char* gw, const TcArgs a) {
  const int d = blockIdx.y;
  if (!((tc_mask >> d) & 1u)) return;
  const mdseg_sparse_graph g = tab.g[d];
  const int npad = a.nt_f[d];
  const int groups = a.n_tiles_f[d] * n_chunks * 4 * npad;  // (tile, chunk, k-group of 8, row)
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < groups; i += gridDim.x * blockDim.x) {
    const int r = i % npad, kg = (i / npad) % 4, kc = (i / (4 * npad)) % n_chunks, z = i / (4 * npad * n_chunks);
    const int n = z * npad + r;
    uint32_t w[TERMS][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = kc * kKB + kg * 8 + 2 * j;
      float v0 = 0.f, v1 = 0.f;
      if (n < g.C_ds) {
        if (c < tab.C_uni) v0 = g.dense[(int64_t)n * tab.C_uni + c];
        if (c + 1 < tab.C_uni) v1 = g.dense[(int64_t)n * tab.C_uni + c + 1];
      }
      uint32_t o[TERMS];
      Split<TERMS>::pair(v0, v1, fmt, o);
#pragma unroll
      for (int t = 0; t < TERMS; ++t) w[t][j] = o[t];
    }
    unsigned char* chunk = gw + a.g_off[d] + ((int64_t)z * n_chunks + kc) * TERMS * npad * 64;
#pragma unroll
    for (int t = 0; t < TERMS; ++t)
      *reinterpret_cast<uint4*>(chunk + (int64_t)t * npad * 64 + kg * (npad * 16) + r * 16) =
          make_uint4(w[t][0], w[t][1], w[t][2], w[t][3]);
  }
}

// adjoint: B[row = u - u0][k = n] = G_d[n][u]; dataset d holds n_tiles x n_chunks(d) chunks of TERMS x [nt][32 k]
template <int TERMS>
__global__ void __launch_bounds__(256) proj_tc_prep_bwd_kernel(const mdseg_graph_table tab, int n_tiles, int fmt,
                                                               unsigned char* gw, const TcArgs a) {
  const int d = blockIdx.y;
  if (!((a.tc_mask >> d) & 1u)) return;
  const mdseg_sparse_graph g = tab.g[d];
  const int nt = a.nt;
  const int n_chunks = (g.C_ds + kKB - 1) / kKB;
  const int groups = n_tiles * n_chunks * 4 * nt;  // (tile, chunk, k-group of 8, row)
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < groups; i += gridDim.x * blockDim.x) {
    const int r = i % nt, kg = (i / nt) % 4, kc = (i / (4 * nt)) % n_chunks, z = i / (4 * nt * n_chunks);
    const int u = z * nt + r;
    uint32_t w[TERMS][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = kc * kKB + kg * 8 + 2 * j;
      float v0 = 0.f, v1 = 0.f;
      if (u < tab.C_uni) {
        if (n < g.C_ds) v0 = g.dense[(int64_t)n * tab.C_uni + u];
        if (n + 1 < g.C_ds) v1 = g.dense[(int64_t)(n + 1) * tab.C_uni + u];
      }
      uint32_t o[TERMS];
      Split<TERMS>::pair(v0, v1, fmt, o);
#pragma unroll
      for (int t = 0; t < TERMS; ++t) w[t][j] = o[t];
    }
    unsigned char* chunk = gw + a.g_off[d] + ((int64_t)z * n_chunks + kc) * TERMS * nt * 64;
#pragma unroll
    for (int t = 0; t < TERMS; ++t)
      *reinterpret_cast<uint4*>(chunk + (int64_t)t * nt * 64 + kg * (nt * 16) + r * 16) =
          make_uint4(w[t][0], w[t][1], w[t][2], w[t][3]);
  }
}

// ---- main kernel -------------------------------------------------------------------------------------------
// kBwd = false: y[n][p] = sum_c G[n][c] x[c][p]       (T = dtype of x, output fp32)
// kBwd = true : dx[u][p] = sum_n G[n][u] dy[n][p]      (T = dtype of dx, input fp32 planes dyA (+ dyB))
template <typename T, int TERMS, bool kBwd>
__global__ void __launch_bounds__(kTcThreads, kBwd ? 4 : 2) proj_tc_kernel(const __grid_constant__ TcArgs a) {
  // the adjoint has one to eight K chunks per CTA: one stage and four CTAs per SM overlap better than two stages
  constexpr int kNS = kBwd ? 1 : kStagesTc;
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar_b[kNS];    // B chunk landed (bulk copy complete_tx)
  __shared__ __align__(8) uint64_t bar_mma[kNS];  // the MMAs that read the stage have retired
  __shared__ __align__(8) uint64_t bar_acc;             // accumulator complete
  __shared__ uint32_t tmem_base_s;

  const int b = blockIdx.y;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  if (d < 0 || d >= a.n_datasets || !((a.tc_mask >> d) & 1u)) return;  // uniform per CTA
  const int C_ds = a.C_ds[d];
  if (!kBwd && (int)blockIdx.z >= a.n_tiles_f[d]) return;                // uniform per CTA
  const int npad = kBwd ? a.nt : a.nt_f[d];
  const int u0 = (int)blockIdx.z * npad;                                 // first output channel of this N tile
  const int n_all = kBwd ? a.C_uni : C_ds;
  const int n_out = (n_all - u0) < npad ? (n_all - u0) : npad;           // valid output channels
  const int K = kBwd ? C_ds : a.C_uni;
  const int n_chunks = (K + kKB - 1) / kKB;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int row = tid & (kTM - 1), khalf = tid >> 7;  // pixel of the tile, half of the K-chunk
  const long long p = (long long)blockIdx.x * kTM + row;
  const bool p_ok = p < a.hw;

  unsigned char* sA = smem;                                        // [stage][term][4 k-groups][128 rows][16 B]
  unsigned char* sB = smem + (size_t)kNS * a.a_stage_bytes;   // [stage][term][4 k-groups][npad rows][16 B]
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < npad) tmem_cols <<= 1;

  if (tid == 0) {
    for (int s = 0; s < kNS; ++s) { mbar_init(&bar_b[s], 1); mbar_init(&bar_mma[s], 1); }
    mbar_init(&bar_acc, 1);
    mbar_fence_init();
  }
  if (warp == 0) {
    tmem_alloc(&tmem_base_s, tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = tmem_base_s;

  const T* xb = kBwd ? nullptr : (const T*)a.x + (long long)b * a.C_uni * a.hw;
  const float* dA = kBwd ? a.dyA + (long long)b * a.y_cmax * a.hw : nullptr;
  const float* dB = (kBwd && a.dyB) ? a.dyB + (long long)b * a.y_cmax * a.hw : nullptr;
  const uint32_t b_chunk_bytes = (uint32_t)(TERMS * npad * 64);
  const unsigned char* gchunks = a.gw + a.g_off[d] + (size_t)blockIdx.z * n_chunks * b_chunk_bytes;
  const uint32_t idesc = umma_idesc(a.fmt, npad);

  // this thread's 16 channels of a chunk, one chunk ahead in registers so that the HBM latency of chunk kc + 1
  // hides behind the conversion, the hand-over and the stage wait of chunk kc
  float vn[kKB / 2];
  auto load_chunk = [&](int kc) {
#pragma unroll
    for (int j = 0; j < kKB / 2; ++j) {
      const int c = kc * kKB + khalf * (kKB / 2) + j;
      float v = 0.f;
      if (p_ok && c < K) {
        if constexpr (kBwd) {
          v = dA[(long long)c * a.hw + p];
          if (dB) v += dB[(long long)c * a.hw + p];
        } else {
          v = to_f32<T>(xb[(long long)c * a.hw + p]);
        }
      }
      vn[j] = v;
    }
  };
  load_chunk(0);

  for (int kc = 0; kc < n_chunks; ++kc) {
    const int s = kc % kNS;
    const uint32_t use = (uint32_t)(kc / kNS);
    float v[kKB / 2];
#pragma unroll
    for (int j = 0; j < kKB / 2; ++j) v[j] = vn[j];
    if (kc + 1 < n_chunks) load_chunk(kc + 1);
    // the MMAs of chunk kc - kStages have finished reading stage s
    if (kc >= kNS) mbar_wait(&bar_mma[s], (use - 1) & 1u);
    unsigned char* stA = sA + (size_t)s * a.a_stage_bytes;
    unsigned char* stB = sB + (size_t)s * a.b_stage_bytes;
    if (tid == 0) {
      mbar_expect_tx(&bar_b[s], b_chunk_bytes);
      bulk_g2s(stB, gchunks + (size_t)kc * b_chunk_bytes, b_chunk_bytes, &bar_b[s]);
    }
    // A: this thread's pixel, 16 channels -> TERMS x 2 k-groups x 16 bytes
#pragma unroll
    for (int kq = 0; kq < 2; ++kq) {
      const int kg = 2 * khalf + kq;
      uint32_t w[TERMS][4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t o[TERMS];
        Split<TERMS>::pair(v[kq * 8 + 2 * j], v[kq * 8 + 2 * j + 1], a.fmt, o);
#pragma unroll
        for (int t = 0; t < TERMS; ++t) w[t][j] = o[t];
      }
#pragma unroll
      for (int t = 0; t < TERMS; ++t)
        *reinterpret_cast<uint4*>(stA + t * (4 * kTM * 16) + kg * (kTM * 16) + row * 16) =
            make_uint4(w[t][0], w[t][1], w[t][2], w[t][3]);
    }
    // generic-proxy writes -> visible to the tensor core's async proxy, then hand over to the issuing thread
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (tid == 0) {
      mbar_wait(&bar_b[s], use & 1u);
      tc_fence_after();
      const uint32_t aA = smem_u32(stA), aB = smem_u32(stB);
#pragma unroll
      for (int ks = 0; ks < kKB / 16; ++ks) {
        // products in order of decreasing weight; TERMS == 1: just (0, 0)
        constexpr int kPairs = TERMS == 3 ? 6 : 1;
        const int ta[6] = {0, 0, 1, 1, 0, 2};
        const int tb[6] = {0, 1, 0, 1, 2, 0};
#pragma unroll
        for (int q = 0; q < kPairs; ++q) {
          const uint64_t ad = umma_desc(aA + ta[q] * (4 * kTM * 16) + ks * 2 * (kTM * 16), kTM * 16, 128, kNoSwizzle);
          const uint64_t bd = umma_desc(aB + tb[q] * (npad * 64) + ks * 2 * (npad * 16), npad * 16, 128, kNoSwizzle);
          umma_f16(tmem_d, ad, bd, idesc, (kc > 0 || ks > 0 || q > 0) ? 1u : 0u);
        }
      }
      tc_commit(&bar_mma[s]);                       // frees the stage when these MMAs retire
      if (kc == n_chunks - 1) tc_commit(&bar_acc);  // ... and the accumulator is complete
    }
  }

  // epilogue: warp w reads TMEM lanes 32(w % 4) .. +31 (= pixels of this tile); the two warps that share a lane
  // quarter take alternate groups of 16 columns
  mbar_wait(&bar_acc, 0);
  tc_fence_after();
  float* yb = kBwd ? nullptr : a.y + ((long long)b * a.y_cmax + u0) * a.hw;
  T* dxb = kBwd ? (T*)a.dx + ((long long)b * a.C_uni + u0) * a.hw : nullptr;
  for (int n0 = (warp >> 2) * 16; n0 < npad; n0 += 32) {
    float acc[16];
    tmem_ld16_f32(tmem_d + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)n0, acc);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (p_ok && n0 + i < n_out) {
        if constexpr (kBwd) dxb[(long long)(n0 + i) * a.hw + p] = from_f32<T>(acc[i]);
        else yb[(long long)(n0 + i) * a.hw + p] = acc[i];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_d, tmem_cols);
}

constexpr int kMaxClasses = 1024;  // forward: up to four N tiles of 256

bool tc_dataset(const mdseg_sparse_graph& g, int C_uni) {
  return g.dense != nullptr && g.C_ds >= 8 && g.C_ds <= kMaxClasses && C_uni >= 32;
}
// forward N tiling of C_ds classes: equal tiles of at most kMaxN rows
void fwd_tiling(int C_ds, int* n_tiles, int* nt) {
  *n_tiles = (pad16(C_ds) + kMaxN - 1) / kMaxN;
  *nt = pad16((C_ds + *n_tiles - 1) / *n_tiles);
}
int terms_of(int dtype) { return dtype == MDSEG_F32 ? 3 : 1; }

}  // namespace
}  // namespace mdseg

extern "C" size_t mdseg_proj_fwd_tc_workspace_bytes(const mdseg_graph_table* graphs, int dtype) {
  using namespace mdseg;
  if (!graph_header_ok(graphs)) return 256;
  const int n_chunks = (graphs->C_uni + kKB - 1) / kKB;
  size_t total = 256;
  for (int i = 0; i < graphs->n_datasets; ++i)
    if (tc_dataset(graphs->g[i], graphs->C_uni)) {
      int n_tiles, nt;
      fwd_tiling(graphs->g[i].C_ds, &n_tiles, &nt);
      total += (size_t)n_tiles * n_chunks * terms_of(dtype) * nt * 64;
    }
  return total;
}

extern "C" int mdseg_proj_fwd_tc(const void* x, int dtype, const mdseg_graph_table* graphs, const int32_t* dataset_ids,
                                 int n_images, int h, int w, float* y, int y_cmax, float* cmax_out, void* workspace,
                                 size_t workspace_bytes, int32_t* err_flag, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(graph_header_ok(graphs), "mdseg_proj_fwd_tc: bad graph table");
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0, "mdseg_proj_fwd_tc: bad shape");
  MDSEG_REQUIRE(is_float_dtype(dtype), "mdseg_proj_fwd_tc: unsupported dtype %d", dtype);
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(x && y && workspace, "mdseg_proj_fwd_tc: null pointer");
  MDSEG_REQUIRE(workspace_bytes >= mdseg_proj_fwd_tc_workspace_bytes(graphs, dtype),
                "mdseg_proj_fwd_tc: workspace too small");
  cudaStream_t s = (cudaStream_t)stream;

  TcArgs a;
  a.x = x; a.y = y; a.dataset_ids = dataset_ids;
  a.gw = reinterpret_cast<unsigned char*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  a.n_datasets = graphs->n_datasets; a.C_uni = graphs->C_uni; a.y_cmax = y_cmax;
  a.hw = (long long)h * w;
  a.n_chunks = (graphs->C_uni + kKB - 1) / kKB;
  a.fmt = dtype == MDSEG_F16 ? 0 : 1;
  a.dyA = nullptr; a.dyB = nullptr; a.dx = nullptr; a.nt = 0;
  const int terms = terms_of(dtype);
  a.tc_mask = 0;
  int npad_max = 0, tiles_max = 1, groups_max = 0;
  long long off = 0;
  for (int i = 0; i < MDSEG_MAX_DATASETS; ++i) {
    a.g_off[i] = 0; a.C_ds[i] = 0; a.nt_f[i] = 0; a.n_tiles_f[i] = 0;
    if (i >= graphs->n_datasets) continue;
    a.C_ds[i] = graphs->g[i].C_ds;
    if (!tc_dataset(graphs->g[i], graphs->C_uni)) continue;
    MDSEG_REQUIRE(y_cmax >= graphs->g[i].C_ds, "mdseg_proj_fwd_tc: y_cmax %d < C_ds %d", y_cmax, graphs->g[i].C_ds);
    a.tc_mask |= 1u << i;
    a.g_off[i] = off;
    fwd_tiling(graphs->g[i].C_ds, &a.n_tiles_f[i], &a.nt_f[i]);
    off += (long long)a.n_tiles_f[i] * a.n_chunks * terms * a.nt_f[i] * 64;
    npad_max = a.nt_f[i] > npad_max ? a.nt_f[i] : npad_max;
    tiles_max = a.n_tiles_f[i] > tiles_max ? a.n_tiles_f[i] : tiles_max;
    const int groups = a.n_tiles_f[i] * a.n_chunks * 4 * a.nt_f[i];
    groups_max = groups > groups_max ? groups : groups_max;
  }
  // sparse graphs and dense ones outside the tensor-core envelope: the CSR / FFMA kernels of proj.cu
  if (int rc = proj_fwd_rest(x, dtype, graphs, dataset_ids, n_images, h, w, y, y_cmax, cmax_out, err_flag, a.tc_mask, s))
    return rc;
  if (!a.tc_mask) return 0;

  a.a_stage_bytes = terms * 4 * kTM * 16;
  a.b_stage_bytes = terms * npad_max * 64;
  const size_t smem = (size_t)kStagesTc * (a.a_stage_bytes + a.b_stage_bytes);
  const dim3 pgrid((unsigned)((groups_max + 255) / 256), (unsigned)graphs->n_datasets);
  const dim3 grid((unsigned)((a.hw + kTM - 1) / kTM), (unsigned)n_images, (unsigned)tiles_max);
  return with_float_type(dtype, "mdseg_proj_fwd_tc", "dtype", [&](auto t) {
    using T = typename decltype(t)::type;
    constexpr int kTerms = std::is_same_v<T, float> ? 3 : 1;
    proj_tc_prep_kernel<kTerms><<<pgrid, 256, 0, s>>>(*graphs, a.tc_mask, a.n_chunks, a.fmt,
                                                      const_cast<unsigned char*>(a.gw), a);
    MDSEG_LAUNCH_OK();
    auto k = proj_tc_kernel<T, kTerms, false>;
    MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<grid, kTcThreads, smem, s>>>(a);
    MDSEG_LAUNCH_OK();
    return 0;
  });
}

// ---- adjoint on the tensor cores ---------------------------------------------------------------------------
namespace mdseg {
int proj_bwd_rest(const float* dyA, const float* dyB, int y_cmax, const mdseg_graph_table* graphs,
                  const int32_t* dataset_ids, int n_images, int h, int w, void* dx, int dtype, unsigned skip_mask,
                  cudaStream_t s);
namespace {
// N tiling of the unified channels: tiles of at most 128 (four CTAs of 48 KB and 128 TMEM columns per SM)
void bwd_tiling(int C_uni, int* n_tiles, int* nt) {
  *n_tiles = (C_uni + 127) / 128;
  *nt = pad16((C_uni + *n_tiles - 1) / *n_tiles);
}
}  // namespace
}  // namespace mdseg

extern "C" size_t mdseg_proj_bwd_tc_workspace_bytes(const mdseg_graph_table* graphs, int dtype) {
  using namespace mdseg;
  if (!graph_header_ok(graphs)) return 256;
  int n_tiles, nt;
  bwd_tiling(graphs->C_uni, &n_tiles, &nt);
  size_t total = 256;
  for (int i = 0; i < graphs->n_datasets; ++i)
    if (tc_dataset(graphs->g[i], graphs->C_uni))
      total += (size_t)n_tiles * ((graphs->g[i].C_ds + kKB - 1) / kKB) * terms_of(dtype) * nt * 64;
  return total;
}

extern "C" int mdseg_proj_bwd_tc(const float* dyA, const float* dyB, int y_cmax, const mdseg_graph_table* graphs,
                                 const int32_t* dataset_ids, int n_images, int h, int w, void* dx, int dtype,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(graph_header_ok(graphs), "mdseg_proj_bwd_tc: bad graph table");
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0, "mdseg_proj_bwd_tc: bad shape");
  MDSEG_REQUIRE(is_float_dtype(dtype), "mdseg_proj_bwd_tc: unsupported dtype %d", dtype);
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(dyA && dx && workspace, "mdseg_proj_bwd_tc: null pointer");
  MDSEG_REQUIRE(workspace_bytes >= mdseg_proj_bwd_tc_workspace_bytes(graphs, dtype),
                "mdseg_proj_bwd_tc: workspace too small");
  cudaStream_t s = (cudaStream_t)stream;

  TcArgs a;
  a.x = nullptr; a.y = nullptr; a.dataset_ids = dataset_ids;
  a.gw = reinterpret_cast<unsigned char*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  a.n_datasets = graphs->n_datasets; a.C_uni = graphs->C_uni; a.y_cmax = y_cmax;
  a.hw = (long long)h * w;
  a.n_chunks = 0;
  a.fmt = dtype == MDSEG_F16 ? 0 : 1;
  a.dyA = dyA; a.dyB = dyB; a.dx = dx;
  int n_tiles;
  bwd_tiling(graphs->C_uni, &n_tiles, &a.nt);
  const int terms = terms_of(dtype);
  a.tc_mask = 0;
  long long off = 0;
  int max_groups = 0;
  for (int i = 0; i < MDSEG_MAX_DATASETS; ++i) {
    a.g_off[i] = 0; a.C_ds[i] = 0; a.nt_f[i] = 0; a.n_tiles_f[i] = 0;
    if (i >= graphs->n_datasets) continue;
    a.C_ds[i] = graphs->g[i].C_ds;
    if (!tc_dataset(graphs->g[i], graphs->C_uni)) continue;
    MDSEG_REQUIRE(y_cmax >= graphs->g[i].C_ds, "mdseg_proj_bwd_tc: y_cmax %d < C_ds %d", y_cmax, graphs->g[i].C_ds);
    a.tc_mask |= 1u << i;
    a.g_off[i] = off;
    const int nch = (graphs->g[i].C_ds + kKB - 1) / kKB;
    off += (long long)n_tiles * nch * terms * a.nt * 64;
    max_groups = n_tiles * nch * 4 * a.nt > max_groups ? n_tiles * nch * 4 * a.nt : max_groups;
  }
  // sparse graphs, dense ones outside the envelope and the zero fill of images without a dataset: proj.cu
  if (int rc = proj_bwd_rest(dyA, dyB, y_cmax, graphs, dataset_ids, n_images, h, w, dx, dtype, a.tc_mask, s)) return rc;
  if (!a.tc_mask) return 0;

  a.a_stage_bytes = terms * 4 * kTM * 16;
  a.b_stage_bytes = terms * a.nt * 64;
  const size_t smem = (size_t)(a.a_stage_bytes + a.b_stage_bytes);  // one stage (kNS == 1 in the adjoint)
  const dim3 pgrid((unsigned)((max_groups + 255) / 256), (unsigned)graphs->n_datasets);
  const dim3 grid((unsigned)((a.hw + kTM - 1) / kTM), (unsigned)n_images, (unsigned)n_tiles);
  return with_float_type(dtype, "mdseg_proj_bwd_tc", "dtype", [&](auto t) {
    using T = typename decltype(t)::type;
    constexpr int kTerms = std::is_same_v<T, float> ? 3 : 1;
    proj_tc_prep_bwd_kernel<kTerms><<<pgrid, 256, 0, s>>>(*graphs, n_tiles, a.fmt, const_cast<unsigned char*>(a.gw), a);
    MDSEG_LAUNCH_OK();
    auto k = proj_tc_kernel<T, kTerms, true>;
    MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<grid, kTcThreads, smem, s>>>(a);
    MDSEG_LAUNCH_OK();
    return 0;
  });
}

// ---- d bi_graph on the tensor cores ------------------------------------------------------------------------
//   dG_d[n][c] += sum over the images b of dataset d and the pixels p of  (dyA + dyB)[b][n][p] * x[b][c][p]
// GEMM per CTA: D[M = 128 classes (one of at most two M tiles), N = C_uni padded to 16 (<= 384, issued as N tiles
// of <= 256; 512 TMEM columns allocated)] over K = one slab of the image's pixels.  Both operands are K-major in HBM already (pixels
// are contiguous), so a thread copies 8 consecutive pixels of one row (32 bytes of fp32), converts them to the 16-bit
// terms and writes one 16-byte K-group per term.  Every element of dy and x is read and converted once per M tile.
// The CTA's 128 x Npad accumulator goes to a slot of the workspace; proj_tc_dgraph_reduce_kernel adds the slots of
// a dataset in a fixed order (deterministic, no atomics).
namespace mdseg {
int proj_dgraph_rest(const void* x, int dtype, const float* dyA, const float* dyB, int y_cmax,
                     const mdseg_graph_table* graphs, const int32_t* dataset_ids, int n_images, int h, int w, float* dG,
                     long long dg_stride, unsigned skip_mask, cudaStream_t s);
namespace {

constexpr int kDgM = 128;        // classes per M tile
constexpr int kDgMaxN = 384;     // unified channels (padded): (128 + 384) rows x 4 K-groups = 8 items per thread
constexpr int kDgItems = 8;      // (row, K-group) items per thread and chunk

struct DgArgs {
  const void* x;
  const float* dyA;
  const float* dyB;
  const int32_t* dataset_ids;
  float* part;                 // [n_images][n_mt M tiles][n_nt N tiles][n_slabs][128][npad]
  int C_ds[MDSEG_MAX_DATASETS];
  unsigned tc_mask;
  int n_datasets, C_uni, npad, y_cmax;  // npad: width of one N tile of unified channels (multiple of 16, <= 384)
  int n_mt, n_nt;              // M tiles of 128 classes (grid), N tiles of npad unified channels
  long long hw, slab;
  int n_slabs, fmt;
  int a_stage_bytes, b_stage_bytes;
};

template <typename T, int TERMS>
__global__ void __launch_bounds__(kTcThreads, 1) proj_tc_dgraph_kernel(const __grid_constant__ DgArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar_mma[kStagesTc];
  __shared__ __align__(8) uint64_t bar_acc;
  __shared__ uint32_t tmem_base_s;

  const int b = blockIdx.z, mt = (int)blockIdx.y % a.n_mt, nz = (int)blockIdx.y / a.n_mt, sl = blockIdx.x;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  if (d < 0 || d >= a.n_datasets || !((a.tc_mask >> d) & 1u)) return;
  const int C_ds = a.C_ds[d];
  const int n0 = mt * kDgM;
  if (n0 >= C_ds) return;
  const int npad = a.npad;
  const int c0x = nz * npad;   // first unified channel of this N tile
  const int R = kDgM + npad;  // rows staged per chunk: 128 of dy, npad of x
  const int tid = threadIdx.x, warp = tid >> 5;
  const long long p_beg = (long long)sl * a.slab;
  const long long p_end = (p_beg + a.slab < a.hw) ? p_beg + a.slab : a.hw;
  const int n_chunks = (int)((p_end - p_beg + kKB - 1) / kKB);

  unsigned char* sA = smem;                                       // [stage][term][4 k-groups][128 rows][16 B]
  unsigned char* sB = smem + (size_t)kStagesTc * a.a_stage_bytes;  // [stage][term][4 k-groups][npad rows][16 B]
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < npad) tmem_cols <<= 1;

  if (tid == 0) {
    for (int s = 0; s < kStagesTc; ++s) mbar_init(&bar_mma[s], 1);
    mbar_init(&bar_acc, 1);
    mbar_fence_init();
  }
  if (warp == 0) {
    tmem_alloc(&tmem_base_s, tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = tmem_base_s;

  const T* xb = (const T*)a.x + (long long)b * a.C_uni * a.hw;
  const float* dA = a.dyA + (long long)b * a.y_cmax * a.hw;
  const float* dB = a.dyB ? a.dyB + (long long)b * a.y_cmax * a.hw : nullptr;
  const bool vec_ok = (a.hw % 8 == 0) && (p_beg % 8 == 0);  // 8 consecutive pixels are 32-byte aligned in every row

  // This thread's (row, K-group) items — the same for every chunk: consecutive threads take consecutive rows of one
  // K-group (conflict-free 16-byte shared-memory stores; a 32-byte sector of HBM per thread and load).
  const int n_items = R * 4;  // <= kDgItems * kTcThreads (npad <= 384)
  const float* srcA[kDgItems];  // dy rows: plane A (and B at the same offset)
  const T* srcX[kDgItems];      // x rows
  int dst_off[kDgItems], kind[kDgItems];  // kind: 0 = none / zero row, 1 = dy row, 2 = x row
#pragma unroll
  for (int j = 0; j < kDgItems; ++j) {
    const int it = j * kTcThreads + tid;
    srcA[j] = nullptr; srcX[j] = nullptr; dst_off[j] = -1; kind[j] = 0;
    if (it < n_items) {
      const int r = it % R, kg = it / R;
      if (r < kDgM) {
        dst_off[j] = kg * (kDgM * 16) + r * 16;
        if (n0 + r < C_ds) { kind[j] = 1; srcA[j] = dA + (long long)(n0 + r) * a.hw + p_beg + kg * 8; }
      } else {
        dst_off[j] = a.a_stage_bytes * kStagesTc + kg * (npad * 16) + (r - kDgM) * 16;  // relative to sA of stage 0 ...
        if (c0x + r - kDgM < a.C_uni) { kind[j] = 2; srcX[j] = xb + (long long)(c0x + r - kDgM) * a.hw + p_beg + kg * 8; }
      }
    }
  }
  const long long plane_b_off = dB ? (dB - dA) : 0;

  // 8 consecutive pixels of item j in chunk kc (zero beyond the matrices / the slab)
  auto load8 = [&](int j, int kc, float (&v)[8]) {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.f;
    const long long off = (long long)kc * kKB;
    const long long p = p_beg + off + ((j * kTcThreads + tid) / R) * 8;
    if (kind[j] == 1) {
      const float* q = srcA[j] + off;
      if (vec_ok && p + 8 <= p_end) {
        const float4 u0 = *reinterpret_cast<const float4*>(q), u1 = *reinterpret_cast<const float4*>(q + 4);
        v[0] = u0.x; v[1] = u0.y; v[2] = u0.z; v[3] = u0.w; v[4] = u1.x; v[5] = u1.y; v[6] = u1.z; v[7] = u1.w;
        if (dB) {
          const float* q2 = q + plane_b_off;
          const float4 w0 = *reinterpret_cast<const float4*>(q2), w1 = *reinterpret_cast<const float4*>(q2 + 4);
          v[0] += w0.x; v[1] += w0.y; v[2] += w0.z; v[3] += w0.w; v[4] += w1.x; v[5] += w1.y; v[6] += w1.z; v[7] += w1.w;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (p + i < p_end) v[i] = q[i] + (dB ? q[plane_b_off + i] : 0.f);
      }
    } else if (kind[j] == 2) {
      const T* q = srcX[j] + off;
      if (vec_ok && p + 8 <= p_end) {
        if constexpr (sizeof(T) == 4) {
          const float4 u0 = *reinterpret_cast<const float4*>(q), u1 = *reinterpret_cast<const float4*>(q + 4);
          v[0] = u0.x; v[1] = u0.y; v[2] = u0.z; v[3] = u0.w; v[4] = u1.x; v[5] = u1.y; v[6] = u1.z; v[7] = u1.w;
        } else {
          VecLoad<T, 8>::load(q, v);
        }
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (p + i < p_end) v[i] = to_f32<T>(q[i]);
      }
    }
  };

  const int n_tiles_n = (npad + kMaxN - 1) / kMaxN;
  const int nt_n = pad16((npad + n_tiles_n - 1) / n_tiles_n);  // N tile width of one UMMA (<= 256)

  // one chunk ahead in registers: the HBM latency of chunk kc + 1 hides behind the conversion of chunk kc
  float vn[kDgItems][8];
#pragma unroll
  for (int j = 0; j < kDgItems; ++j) load8(j, 0, vn[j]);

  for (int kc = 0; kc < n_chunks; ++kc) {
    const int s = kc % kStagesTc;
    const uint32_t use = (uint32_t)(kc / kStagesTc);
    float v[kDgItems][8];
#pragma unroll
    for (int j = 0; j < kDgItems; ++j)
#pragma unroll
      for (int i = 0; i < 8; ++i) v[j][i] = vn[j][i];
    if (kc + 1 < n_chunks) {
#pragma unroll
      for (int j = 0; j < kDgItems; ++j) load8(j, kc + 1, vn[j]);
    }
    if (kc >= kStagesTc) mbar_wait(&bar_mma[s], (use - 1) & 1u);
    unsigned char* stA = sA + (size_t)s * a.a_stage_bytes;
    unsigned char* stB = sB + (size_t)s * a.b_stage_bytes;
#pragma unroll
    for (int j = 0; j < kDgItems; ++j) {
      if (dst_off[j] >= 0) {
        uint32_t w[TERMS][4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint32_t o[TERMS];
          Split<TERMS>::pair(v[j][2 * q], v[j][2 * q + 1], a.fmt, o);
#pragma unroll
          for (int t = 0; t < TERMS; ++t) w[t][q] = o[t];
        }
        const bool is_a = dst_off[j] < a.a_stage_bytes * kStagesTc;
        unsigned char* dst = is_a ? stA + dst_off[j] : stB + (dst_off[j] - a.a_stage_bytes * kStagesTc);
        const int tstride = is_a ? 4 * kDgM * 16 : 4 * npad * 16;
#pragma unroll
        for (int t = 0; t < TERMS; ++t)
          *reinterpret_cast<uint4*>(dst + t * tstride) = make_uint4(w[t][0], w[t][1], w[t][2], w[t][3]);
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      const uint32_t aA = smem_u32(stA), aB = smem_u32(stB);
      for (int jn = 0; jn < n_tiles_n; ++jn) {
        const int col0 = jn * nt_n;
        const int nn = (npad - col0) < nt_n ? (npad - col0) : nt_n;
        const uint32_t idesc = umma_idesc(a.fmt, nn);
#pragma unroll
        for (int ks = 0; ks < kKB / 16; ++ks) {
          constexpr int kPairs = TERMS == 3 ? 6 : 1;
          const int ta[6] = {0, 0, 1, 1, 0, 2};
          const int tb[6] = {0, 1, 0, 1, 2, 0};
#pragma unroll
          for (int q = 0; q < kPairs; ++q) {
            const uint64_t ad = umma_desc(aA + ta[q] * (4 * kDgM * 16) + ks * 2 * (kDgM * 16), kDgM * 16, 128, kNoSwizzle);
            const uint64_t bd =
                umma_desc(aB + tb[q] * (4 * npad * 16) + ks * 2 * (npad * 16) + col0 * 16, npad * 16, 128, kNoSwizzle);
            umma_f16(tmem_d + (uint32_t)col0, ad, bd, idesc, (kc > 0 || ks > 0 || q > 0) ? 1u : 0u);
          }
        }
      }
      tc_commit(&bar_mma[s]);
      if (kc == n_chunks - 1) tc_commit(&bar_acc);
    }
  }

  // epilogue: TMEM lane = class row of the M tile, columns = unified channels -> this CTA's slot of the workspace
  mbar_wait(&bar_acc, 0);
  tc_fence_after();
  float* slot = a.part + ((((long long)b * a.n_mt + mt) * a.n_nt + nz) * a.n_slabs + sl) * (long long)kDgM * npad;
  const int row = (warp & 3) * 32 + (tid & 31);
  for (int c0 = (warp >> 2) * 16; c0 < npad; c0 += 32) {
    float acc[16];
    tmem_ld16_f32(tmem_d + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)c0, acc);
    float4* o = reinterpret_cast<float4*>(slot + (long long)row * npad + c0);
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = make_float4(acc[4 * i], acc[4 * i + 1], acc[4 * i + 2], acc[4 * i + 3]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_d, tmem_cols);
}

// dG[d][n][c] += sum of the slots of dataset d in (image, slab) order
__global__ void __launch_bounds__(256) proj_tc_dgraph_reduce_kernel(const DgArgs a, int n_images, float* __restrict__ dG,
                                                                    long long dg_stride) {
  const int d = blockIdx.y;
  if (!((a.tc_mask >> d) & 1u)) return;
  const int C_ds = a.C_ds[d];
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= C_ds * a.C_uni) return;
  const int n = idx / a.C_uni, c = idx - n * a.C_uni;
  const int mt = n / kDgM, r = n - mt * kDgM;
  const int nz = c / a.npad, cc = c - nz * a.npad;
  float sum = 0.f;
  for (int b = 0; b < n_images; ++b) {
    if ((a.dataset_ids ? a.dataset_ids[b] : 0) != d) continue;
    const float* base = a.part + ((((long long)b * a.n_mt + mt) * a.n_nt + nz) * a.n_slabs) * (long long)kDgM * a.npad +
                        (long long)r * a.npad + cc;
    for (int sl = 0; sl < a.n_slabs; ++sl) sum += base[(long long)sl * kDgM * a.npad];
  }
  dG[(long long)d * dg_stride + idx] += sum;
}

bool dg_dataset(const mdseg_sparse_graph& g, int C_uni) { return tc_dataset(g, C_uni) && C_uni <= 4 * kDgMaxN; }
// N tiling of the unified channels: equal tiles of at most kDgMaxN
void dg_tiling(int C_uni, int* n_nt, int* npad) {
  *n_nt = (pad16(C_uni) + kDgMaxN - 1) / kDgMaxN;
  *npad = pad16((C_uni + *n_nt - 1) / *n_nt);
}
int dg_m_tiles(const mdseg_graph_table* graphs) {
  int m = 1;
  for (int i = 0; i < graphs->n_datasets; ++i)
    if (dg_dataset(graphs->g[i], graphs->C_uni)) {
      const int t = (graphs->g[i].C_ds + kDgM - 1) / kDgM;
      m = t > m ? t : m;
    }
  return m;
}

int dg_slabs(int n_images, long long hw) {
  long long n = (2LL * sm_count() + n_images - 1) / n_images;  // about two CTAs' worth of work per SM
  const long long max_slabs = (hw + 1023) / 1024;              // at least 1024 pixels (32 chunks) per CTA
  if (n > max_slabs) n = max_slabs;
  if (n < 1) n = 1;
  return (int)n;
}

}  // namespace
}  // namespace mdseg

extern "C" size_t mdseg_proj_bwd_graph_tc_workspace_bytes(const mdseg_graph_table* graphs, int n_images, int h, int w) {
  using namespace mdseg;
  if (!graphs || graphs->C_uni <= 0 || n_images <= 0 || h <= 0 || w <= 0) return 256;
  const int n_slabs = dg_slabs(n_images, (long long)h * w);
  int n_nt, npad;
  dg_tiling(graphs->C_uni, &n_nt, &npad);
  return (size_t)n_images * dg_m_tiles(graphs) * n_nt * n_slabs * kDgM * npad * 4 + 512;
}

extern "C" int mdseg_proj_bwd_graph_tc(const void* x, int dtype, const float* dyA, const float* dyB, int y_cmax,
                                       const mdseg_graph_table* graphs, const int32_t* dataset_ids, int n_images, int h,
                                       int w, float* dG, long long dg_stride, void* workspace, size_t workspace_bytes,
                                       void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(graph_header_ok(graphs), "mdseg_proj_bwd_graph_tc: bad graph table");
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0, "mdseg_proj_bwd_graph_tc: bad shape");
  MDSEG_REQUIRE(is_float_dtype(dtype), "mdseg_proj_bwd_graph_tc: unsupported dtype %d", dtype);
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(x && dyA && dG && workspace, "mdseg_proj_bwd_graph_tc: null pointer");
  MDSEG_REQUIRE(workspace_bytes >= mdseg_proj_bwd_graph_tc_workspace_bytes(graphs, n_images, h, w),
                "mdseg_proj_bwd_graph_tc: workspace too small");
  cudaStream_t s = (cudaStream_t)stream;

  DgArgs a;
  a.x = x; a.dyA = dyA; a.dyB = dyB; a.dataset_ids = dataset_ids;
  a.part = reinterpret_cast<float*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  a.n_datasets = graphs->n_datasets; a.C_uni = graphs->C_uni; a.y_cmax = y_cmax;
  dg_tiling(graphs->C_uni, &a.n_nt, &a.npad);
  a.n_mt = dg_m_tiles(graphs);
  a.hw = (long long)h * w;
  a.n_slabs = dg_slabs(n_images, a.hw);
  a.slab = ((a.hw + a.n_slabs - 1) / a.n_slabs + kKB - 1) / kKB * kKB;  // whole chunks, 32-pixel aligned starts
  a.n_slabs = (int)((a.hw + a.slab - 1) / a.slab);
  a.fmt = dtype == MDSEG_F16 ? 0 : 1;
  const int terms = terms_of(dtype);
  a.tc_mask = 0;
  int cmax = 0;
  for (int i = 0; i < MDSEG_MAX_DATASETS; ++i) {
    a.C_ds[i] = i < graphs->n_datasets ? graphs->g[i].C_ds : 0;
    if (i < graphs->n_datasets && dg_dataset(graphs->g[i], graphs->C_uni)) {
      MDSEG_REQUIRE(y_cmax >= graphs->g[i].C_ds, "mdseg_proj_bwd_graph_tc: y_cmax %d < C_ds %d", y_cmax, graphs->g[i].C_ds);
      MDSEG_REQUIRE(dg_stride >= (long long)graphs->g[i].C_ds * graphs->C_uni, "mdseg_proj_bwd_graph_tc: dg_stride too small");
      a.tc_mask |= 1u << i;
      cmax = graphs->g[i].C_ds > cmax ? graphs->g[i].C_ds : cmax;
    }
  }
  // everything outside the tensor-core envelope: the FFMA kernel of proj.cu
  if (int rc = proj_dgraph_rest(x, dtype, dyA, dyB, y_cmax, graphs, dataset_ids, n_images, h, w, dG, dg_stride, a.tc_mask, s))
    return rc;
  if (!a.tc_mask) return 0;

  a.a_stage_bytes = terms * 4 * kDgM * 16;
  a.b_stage_bytes = terms * 4 * a.npad * 16;
  const size_t smem = (size_t)kStagesTc * (a.a_stage_bytes + a.b_stage_bytes);
  MDSEG_REQUIRE(smem <= 220 * 1024, "mdseg_proj_bwd_graph_tc: C_uni too large for the staged operands");
  const dim3 grid((unsigned)a.n_slabs, (unsigned)(a.n_mt * a.n_nt), (unsigned)n_images);
  const dim3 rgrid((unsigned)(((long long)cmax * a.C_uni + 255) / 256), (unsigned)graphs->n_datasets);
  if (int rc = with_float_type(dtype, "mdseg_proj_bwd_graph_tc", "dtype", [&](auto t) {
        using T = typename decltype(t)::type;
        auto k = proj_tc_dgraph_kernel<T, std::is_same_v<T, float> ? 3 : 1>;
        MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k<<<grid, kTcThreads, smem, s>>>(a);
        MDSEG_LAUNCH_OK();
        return 0;
      }))
    return rc;
  proj_tc_dgraph_reduce_kernel<<<rgrid, 256, 0, s>>>(a, n_images, dG, dg_stride);
  MDSEG_LAUNCH_OK();
  return 0;
}
