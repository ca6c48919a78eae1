// up_ce_warp.cu — warp-private fused bilinear upsample (align_corners=True) + per-pixel CE forward:
// the fast path of mdseg_up_ce_fwd for fp32 low-res logits, uint8 labels and up-sampling
// factors in [1, 5] (the training geometry is stride 4).
// Reference work replaced: F.interpolate(..., mode='bilinear', align_corners=True) of
// lib/loss/loss_cross_datasets.py:1007,1051 + nn.CrossEntropyLoss(ignore_index=255,
// reduction='none') of lib/loss/ohem_ce_loss.py:27,61 and the `loss > thresh` counting of
// ohem_ce_loss.py:25-30 / :52-74.  The [B,C,H,W] upsampled tensor is never materialised.
//
// One WARP per unit (CTA = 32 threads, nothing shared between warps):
//   unit = (image b, strip of 32 low-res cells, segment of `seg_rows` cell-rows), all classes.
//   lane l owns cell x = 32*strip + l: its 4 corners are 4 LDS per class, reused by the 4..5 x 4..5
//   label pixels of the cell, which live in registers.
//   * class planes of low-res rows (g, g+1) arrive as 4-D TMA boxes [8 classes][2 rows][36 cols] in a
//     3-stage mbarrier ring; the channel-maximum rows and the label bytes of the NEXT cell-row are
//     prefetched with bulk copies while the current one is computed;
//   * per (pixel, class): half an FFMA2, one MUFU.EX2, half an FADD2 — the corners are shifted by the
//     per-corner channel maximum first, so the interpolated exponent is <= 0 and no running maximum
//     is needed; the label-class logit is picked with one packed fp16 compare per two pixels;
//   * loss / lse rows leave through a per-warp row buffer as contiguous 4-byte stores; the OHEM
//     counters (n_valid, n_hard, sum_hard, n_px) are reduced in the warp and added with one RED each.
#include "tma_util.cuh"

namespace mdseg {
namespace {

using namespace tma;

constexpr int kKC = 8;                          // classes per TMA stage
constexpr int kBoxW = 36;                       // staged columns: 33 needed, rows of 144 B
#ifndef MDSEG_FWD_STAGES
#define MDSEG_FWD_STAGES 3
#endif
constexpr int kStages = MDSEG_FWD_STAGES;
constexpr int kStageFloats = kKC * 2 * kBoxW;   // 576
constexpr int kStageBytes = kStageFloats * 4;   // 2304
constexpr int kStgW = 176;                      // staged label columns: <= 15 alignment + 32 cells x 5
constexpr int kMaxR = 5;
constexpr int kSpan = 160;

struct Args {
  mdseg_src_table src;
  const int32_t* dataset_ids;
  const uint8_t* labels;
  Geom gm;
  int ignore;
  float* loss_px;
  float* lse_px;
  mdseg_ohem_state* states;
  int* err_flag;
  int seg_rows, n_seg, n_strips;
};

// T := arg where the pixel's class (fp16 pair `lab2`) equals the current class (`c2`)
__device__ __forceinline__ void pick_label2(float2& T, float2 arg, uint32_t lab2, uint32_t c2) {
  asm("{ .reg .pred p, q;\n"
      "  setp.eq.f16x2 p|q, %4, %5;\n"
      "  @p mov.f32 %0, %2;\n"
      "  @q mov.f32 %1, %3; }"
      : "+f"(T.x), "+f"(T.y)
      : "f"(arg.x), "f"(arg.y), "r"(lab2), "r"(c2));
}

struct Unit {
  int lane, b, x0, xl, sx, nx, C, g0, g1, n_ch, n_loads, Xa, wst, Xw0, nw;
  int inv_nch;  // ceil(65536 / n_ch)
  int slot;     // stage of the TMA ring the next chunk arrives in, and its barrier phase
  uint32_t phase;
  bool cell_ok;
};

// lane 0: queue the label bytes and the channel-maximum rows of a cell-row
__device__ __forceinline__ void issue_staging(const Args& a, const Unit& un, const CUtensorMap* cmap, int g, int Ys,
                                              int R, uint8_t* labs, float* cms, uint64_t* sbar) {
  mbar_expect_tx(sbar, (uint32_t)(R * un.wst + 2 * kBoxW * 4));
  for (int j = 0; j < R; ++j) {
    const int64_t p = ((int64_t)un.b * a.gm.H + (Ys + j)) * a.gm.W + un.Xa;
    bulk_g2s(labs + j * kStgW, a.labels + p, (uint32_t)un.wst, sbar);
  }
  load_3d(cms, cmap, sbar, un.x0, g, un.b);
}

template <int RT, bool NX5>
__device__ __forceinline__ void cell_row(const Args& a, const CUtensorMap* map, const CUtensorMap* cmap, Unit& un,
                                         int g, int Ys, int R, int Ys_next, int R_next, const float (&l1w)[5],
                                         const float (&l1h)[kMaxR], float* stages, uint64_t* bars, uint8_t* labs,
                                         float* cms, float* rb, float thresh, unsigned& n_valid, unsigned& n_hard,
                                         unsigned& n_px, float& sum_hard, int& err) {
  const int lane = un.lane;
  // class ids of this lane's pixels as fp16 pairs (255.0 = ignored / invalid: never a class)
  uint32_t LH[RT][2], lh4[RT];
#pragma unroll
  for (int j = 0; j < RT; ++j) {
    uint32_t hv[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      uint32_t v = 255u;
      if (j < R && i < un.nx) {
        v = labs[j * kStgW + un.sx + i];
        if (v != (uint32_t)a.ignore && v >= (uint32_t)un.C) { err |= MDSEG_ERR_LABEL_RANGE; v = 255u; }
        if (v == (uint32_t)a.ignore) v = 255u;
      }
      hv[i] = (uint32_t)__half_as_ushort(__ushort2half_rn((unsigned short)v));
    }
    LH[j][0] = hv[0] | (hv[1] << 16);
    LH[j][1] = hv[2] | (hv[3] << 16);
    lh4[j] = hv[4] | (0x5bf8u << 16);
    // keep the packed form live: under register pressure ptxas otherwise re-packs the halves inside the class loop
    asm volatile("" : "+r"(LH[j][0]), "+r"(LH[j][1]));
  }
  // per-corner channel maxima (already in log2 units), and their interpolation M per pixel column
  const float c00 = cms[un.xl] * kLog2e, c01 = cms[un.xl + 1] * kLog2e;
  const float c10 = cms[kBoxW + un.xl] * kLog2e, c11 = cms[kBoxW + un.xl + 1] * kLog2e;
  __syncwarp();
  if (lane == 0 && g + 1 < un.g1) issue_staging(a, un, cmap, g + 1, Ys_next, R_next, labs, cms, &bars[kStages]);

  float2 L1H[RT];
#pragma unroll
  for (int j = 0; j < RT; ++j) L1H[j] = dup2(l1h[j]);
  const float2 L1W[2] = {make_float2(l1w[0], l1w[1]), make_float2(l1w[2], l1w[3])};
  const float l1w4 = l1w[4];

  float2 S[RT][2], T[RT][2];
  float s4[RT], t4[RT];
#pragma unroll
  for (int j = 0; j < RT; ++j) {
    S[j][0] = S[j][1] = make_float2(0.f, 0.f);
    T[j][0] = T[j][1] = make_float2(0.f, 0.f);
    s4[j] = 0.f; t4[j] = 0.f;
  }

  uint32_t c2 = 0u;  // fp16 pair (0.0, 0.0): the class ids simply keep counting across the chunks of the cell-row
#pragma unroll 1
  for (int k = 0; k < un.n_ch; ++k) {
    const int q = (g - un.g0) * un.n_ch + k;
    const int c_lo = k * kKC;
    const int cc = (un.C - c_lo) < kKC ? (un.C - c_lo) : kKC;
    const int slot = un.slot;          // ring position and phase are carried, not derived from q by division
    mbar_wait(&bars[slot], un.phase);
    if (++un.slot == kStages) { un.slot = 0; un.phase ^= 1u; }
    const float* Sp = stages + slot * kStageFloats + un.xl;
#pragma unroll 1
    for (int c = 0; c < cc; ++c, c2 = next_class2(c2)) {
      // corners, in log2 units, minus the corner's channel maximum: every interpolated exponent is <= 0
      const float v00 = fmaf(Sp[0], kLog2e, -c00), v01 = fmaf(Sp[1], kLog2e, -c01);
      const float v10 = fmaf(Sp[kBoxW], kLog2e, -c10), v11 = fmaf(Sp[kBoxW + 1], kLog2e, -c11);
      Sp += 2 * kBoxW;
      const float dv0 = v01 - v00, dv1 = v11 - v10;
      const float2 V0 = dup2(v00), DV0 = dup2(dv0), V1 = dup2(v10), DV1 = dup2(dv1);
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        const float2 h0 = fma2(L1W[p], DV0, V0);
        const float2 dd = sub2(fma2(L1W[p], DV1, V1), h0);
#pragma unroll
        for (int j = 0; j < RT; ++j) {
          const float2 arg = fma2(L1H[j], dd, h0);
          pick_label2(T[j][p], arg, LH[j][p], c2);
          S[j][p] = add2(S[j][p], ex2_2(arg));
        }
      }
      if (NX5) {
        const float h0 = fmaf(l1w4, dv0, v00);
        const float dd = fmaf(l1w4, dv1, v10) - h0;
#pragma unroll
        for (int j = 0; j < RT; ++j) {
          const float arg = fmaf(l1h[j], dd, h0);
          float2 t = make_float2(t4[j], 0.f);
          pick_label2(t, make_float2(arg, 0.f), lh4[j], c2);
          t4[j] = t.x;
          s4[j] += ex2_approx(arg);
        }
      }
    }
    __syncwarp();
    if (lane == 0 && q + kStages < un.n_loads) {  // the slot is free: every lane has read its corners
      const int qn = q + kStages;
      const int qrow = (qn * un.inv_nch) >> 16;  // qn / n_ch by a 16-bit reciprocal (qn < 128, n_ch <= 32): no division
      const int qk = qn - qrow * un.n_ch;
      mbar_expect_tx(&bars[slot], kStageBytes);
      load_4d(stages + slot * kStageFloats, map, &bars[slot], un.x0, un.g0 + qrow, qk * kKC, un.b);
    }
  }

  // finalize: lse = M + log2(sum), loss = lse - z_label; rows leave through the warp's row buffer
  const float dm0 = c01 - c00, dm1 = c11 - c10;
  const int off = un.sx - (un.Xw0 - un.Xa);
  // straight-line and predicated: this code runs once per cell-row from a cold instruction cache, so every
  // instruction costs several cycles — no per-pixel branches, per-column terms hoisted, 32-bit row offsets
  float hm0[NX5 ? 5 : 4], dhm[NX5 ? 5 : 4];
#pragma unroll
  for (int i = 0; i < (NX5 ? 5 : 4); ++i) {
    hm0[i] = fmaf(l1w[i], dm0, c00);
    dhm[i] = fmaf(l1w[i], dm1, c10) - hm0[i];
  }
  float* lp = a.loss_px + (((int64_t)un.b * a.gm.H + Ys) * a.gm.W + un.Xw0);
  float* ep = a.lse_px + (((int64_t)un.b * a.gm.H + Ys) * a.gm.W + un.Xw0);
  n_px += (unsigned)(R * un.nx);
#pragma unroll
  for (int j = 0; j < RT; ++j) {
    if (j < R) {  // warp-uniform
#pragma unroll
      for (int i = 0; i < (NX5 ? 5 : 4); ++i) {
        const bool on = i < un.nx;
        const float sv = i == 4 ? s4[j] : (i & 1 ? S[j][i >> 1].y : S[j][i >> 1].x);
        const float tv = i == 4 ? t4[j] : (i & 1 ? T[j][i >> 1].y : T[j][i >> 1].x);
        const uint32_t hv = i == 4 ? (lh4[j] & 0xffffu) : ((LH[j][i >> 1] >> (16 * (i & 1))) & 0xffffu);
        const bool valid = hv != 0x5bf8u;
        const float lg = lg2_approx(sv);
        const float l = valid ? (lg - tv) * kLn2 : 0.f;
        const float e = (fmaf(l1h[j], dhm[i], hm0[i]) + lg) * kLn2;
        if (on) { rb[off + i] = l; rb[kSpan + off + i] = e; }
        const bool hard = on && l > thresh;
        n_valid += (on && valid) ? 1u : 0u;
        n_hard += hard ? 1u : 0u;
        sum_hard += hard ? l : 0.f;
      }
      __syncwarp();
#pragma unroll 1
      for (int k = lane; k < un.nw; k += 32) {
        lp[k] = rb[k];
        ep[k] = rb[kSpan + k];
      }
      lp += a.gm.W;
      ep += a.gm.W;
      __syncwarp();
    }
  }
}

constexpr size_t kOffCm = (size_t)kStages * kStageBytes;
constexpr size_t kOffLab = kOffCm + 2 * kBoxW * 4;
constexpr size_t kOffRb = kOffLab + (size_t)kMaxR * kStgW;
constexpr size_t kOffBars = kOffRb + 2 * kSpan * 4;
constexpr size_t kSmem = kOffBars + (kStages + 1) * 8;
static_assert(kOffCm % 128 == 0 && kOffLab % 16 == 0 && kOffRb % 16 == 0 && kOffBars % 8 == 0, "smem carve-up");

#ifndef MDSEG_FWD_OCC
#define MDSEG_FWD_OCC 14
#endif
__global__ void __launch_bounds__(32, MDSEG_FWD_OCC) up_ce_fwd_warp_kernel(const __grid_constant__ Maps maps,
                                                                const __grid_constant__ CUtensorMap cmap,
                                                                const __grid_constant__ Args a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* stages = reinterpret_cast<float*>(smem_raw);
  uint8_t* labs = smem_raw + kOffLab;                            // [kMaxR][kStgW]
  float* cms = reinterpret_cast<float*>(smem_raw + kOffCm);      // [2][kBoxW] channel maxima of rows g, g+1
  float* rb = reinterpret_cast<float*>(smem_raw + kOffRb);       // [2][kSpan] loss / lse row
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + kOffBars);

  const Geom& gm = a.gm;
  const int lane = threadIdx.x;
  const int b = blockIdx.y;
  const int strip = blockIdx.x % a.n_strips, seg = blockIdx.x / a.n_strips;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  const int h = gm.h, w = gm.w;
  const int x0 = strip * 32;
  const int x = x0 + lane;
  const int g0 = seg * a.seg_rows;
  const int g1 = (g0 + a.seg_rows < h - 1) ? g0 + a.seg_rows : h - 1;

  // horizontal geometry of this lane's cell
  const bool cell_ok = x <= w - 2;
  int Xbeg = 0, Xend = 0;
  if (cell_ok) cell_span(gm.xm, x, gm.W, Xbeg, Xend);
  const int nx = Xend - Xbeg;
  const unsigned cmask = __ballot_sync(0xffffffffu, cell_ok);
  const int Xw0 = __shfl_sync(0xffffffffu, Xbeg, 0);
  const int Xw1 = __shfl_sync(0xffffffffu, Xend, 31 - __clz(cmask));
  // label-row range of every cell-row of the segment: lane t holds the first label row of cell-row g0 + t
  int ys_tab = gm.H;
  if (g0 + lane < h - 1) ys_tab = first_dst_ge(gm.ym, g0 + lane, gm.H);

  if (d < 0 || d >= a.src.n_datasets) {
    // image outside every dataset: not part of the loss vector (sentinel -1), but its labels still
    // count in n_min (ohem_ce_loss.py:52 uses all labels)
    const int Ya = __shfl_sync(0xffffffffu, ys_tab, 0), Yb = __shfl_sync(0xffffffffu, ys_tab, g1 - g0);
    unsigned nv = 0;
    for (int Y = Ya; Y < Yb; ++Y)
      for (int k = lane; k < Xw1 - Xw0; k += 32) {
        const int64_t p = ((int64_t)b * gm.H + Y) * gm.W + Xw0 + k;
        a.loss_px[p] = -1.0f;
        a.lse_px[p] = 0.f;
        nv += ((int)a.labels[p] != a.ignore) ? 1u : 0u;
      }
    nv = warp_sum(nv);
    if (lane == 0) {
      if (nv) atomicAdd(&a.states->n_valid, (unsigned long long)nv);
      if (blockIdx.x == 0) atomicOr(a.err_flag, MDSEG_ERR_DATASET_ID);
    }
    return;
  }

  Unit un;
  un.lane = lane; un.b = b; un.x0 = x0; un.xl = cell_ok ? lane : 0; un.nx = nx; un.C = a.src.C[d];
  un.g0 = g0; un.g1 = g1; un.cell_ok = cell_ok;
  un.n_ch = (un.C + kKC - 1) / kKC;
  un.n_loads = (g1 - g0) * un.n_ch;
  un.inv_nch = (65536 + un.n_ch - 1) / un.n_ch;
  un.slot = 0; un.phase = 0u;
  un.Xw0 = Xw0; un.nw = Xw1 - Xw0;
  un.Xa = Xw0 & ~15;
  un.sx = cell_ok ? Xbeg - un.Xa : 0;
  un.wst = (gm.W - un.Xa) < kStgW ? (gm.W - un.Xa) : kStgW;
  const CUtensorMap* map = &maps.m[d];
  mdseg_ohem_state* st = a.states + (a.src.seg_per_dataset ? d : 0);
  const float thresh = st->thresh;

  if (lane == 0) {
    prefetch_map(map);
    prefetch_map(&cmap);
    for (int s = 0; s <= kStages; ++s) mbar_init(&bars[s], 1);
    mbar_fence_init();
    {
      int Ys0, Ye0;
      cell_span(gm.ym, g0, gm.H, Ys0, Ye0);
      issue_staging(a, un, &cmap, g0, Ys0, Ye0 - Ys0, labs, cms, &bars[kStages]);
    }
    for (int qn = 0; qn < kStages && qn < un.n_loads; ++qn) {
      mbar_expect_tx(&bars[qn], kStageBytes);
      load_4d(stages + qn * kStageFloats, map, &bars[qn], x0, g0 + qn / un.n_ch, (qn % un.n_ch) * kKC, b);
    }
  }
  float l1w[5];
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    int cell;
    l1w[i] = 0.f;
    if (i < nx) axis_cell(gm.xm, Xbeg + i, cell, l1w[i]);
  }
  const bool nx5 = __any_sync(0xffffffffu, nx > 4);
  __syncwarp();

  unsigned n_valid = 0, n_hard = 0, n_px = 0;
  float sum_hard = 0.f;
  int err = 0;
  for (int g = g0; g < g1; ++g) {
    const int Ys = __shfl_sync(0xffffffffu, ys_tab, g - g0);
    const int Ye = __shfl_sync(0xffffffffu, ys_tab, g - g0 + 1);
    const int Rn = __shfl_sync(0xffffffffu, ys_tab, (g - g0 + 2) & 31) - Ye;
    const int R = Ye - Ys;
    float l1h[kMaxR];
#pragma unroll
    for (int j = 0; j < kMaxR; ++j) {
      int cell;
      l1h[j] = 0.f;
      if (j < R) axis_cell(gm.ym, Ys + j, cell, l1h[j]);
    }
    mbar_wait(&bars[kStages], (uint32_t)((g - g0) & 1));
#define MDSEG_ROW(RT, N5)                                                                                          \
  cell_row<RT, N5>(a, map, &cmap, un, g, Ys, R, Ye, Rn, l1w, l1h, stages, bars, labs, cms, rb, thresh, n_valid, n_hard, \
                   n_px, sum_hard, err)
    if (R <= 4) {
      if (nx5) MDSEG_ROW(4, true); else MDSEG_ROW(4, false);
    } else {
      if (nx5) MDSEG_ROW(5, true); else MDSEG_ROW(5, false);
    }
#undef MDSEG_ROW
  }

  n_valid = warp_sum(n_valid);
  n_hard = warp_sum(n_hard);
  n_px = warp_sum(n_px);
  const double sh = warp_sum((double)sum_hard);
  if (__any_sync(0xffffffffu, err != 0) && lane == 0) atomicOr(a.err_flag, MDSEG_ERR_LABEL_RANGE);
  if (lane == 0) {
    if (n_valid) atomicAdd(&st->n_valid, (unsigned long long)n_valid);
    if (n_hard) { atomicAdd(&st->n_hard, (unsigned long long)n_hard); atomicAdd(&st->sum_hard, sh); }
    if (n_px) atomicAdd(&st->n_px, (unsigned long long)n_px);
  }
}

}  // namespace

// Return 0 = launched, -1 = not applicable (caller falls back), > 0 = error.
int up_ce_fwd_warp(const FwdArgs& fa, int label_dtype, int n_images, cudaStream_t s) {
  if (label_dtype != MDSEG_U8 || fa.src.cmax == nullptr) return -1;
  if (fa.gm.W % 16 != 0 || ((uintptr_t)fa.labels & 15) != 0 || ((uintptr_t)fa.src.cmax & 15) != 0) return -1;
  if (fa.ignore < 0 || fa.ignore > 255) return -1;
  if (!tma::fast_geometry(fa.src, fa.gm)) return -1;
  tma::Maps maps;
  if (int rc = tma::make_maps(fa.src, fa.gm, n_images, kBoxW, 2, kKC, &maps)) return rc;
  if (!fa.src.cmax_ready)  // aux heads: nobody produced the channel maximum yet
    if (int rc = tma::channel_max(fa.src, fa.dataset_ids, n_images, (int64_t)fa.gm.h * fa.gm.w, s)) return rc;
  CUtensorMap cmap;
  {
    const tma::EncodeTiledFn enc = tma::encode_fn();
    if (!enc) return -1;
    cuuint64_t dims[3] = {(cuuint64_t)fa.gm.w, (cuuint64_t)fa.gm.h, (cuuint64_t)n_images};
    cuuint64_t strides[2] = {(cuuint64_t)fa.gm.w * 4, (cuuint64_t)fa.gm.h * fa.gm.w * 4};
    cuuint32_t box[3] = {(cuuint32_t)kBoxW, 2, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(&cmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, fa.src.cmax, dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("cuTensorMapEncodeTiled failed for the channel-maximum plane (CUresult %d)", (int)r);
      return 1;
    }
  }
  Args a;
  a.src = fa.src; a.dataset_ids = fa.dataset_ids; a.labels = (const uint8_t*)fa.labels; a.gm = fa.gm;
  a.ignore = fa.ignore; a.loss_px = fa.loss_px; a.lse_px = fa.lse_px; a.states = fa.states; a.err_flag = fa.err_flag;
#ifndef MDSEG_FWD_SEG_ROWS
#define MDSEG_FWD_SEG_ROWS 2
#endif
  a.seg_rows = fa.gm.h - 1 < MDSEG_FWD_SEG_ROWS ? fa.gm.h - 1 : MDSEG_FWD_SEG_ROWS;
  a.n_seg = (fa.gm.h - 1 + a.seg_rows - 1) / a.seg_rows;
  a.n_strips = (fa.gm.w - 1 + 31) / 32;
  MDSEG_CUDA_OK(cudaFuncSetAttribute(up_ce_fwd_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem));
  dim3 grid((unsigned)(a.n_strips * a.n_seg), (unsigned)n_images);
  up_ce_fwd_warp_kernel<<<grid, 32, kSmem, s>>>(maps, cmap, a);
  MDSEG_LAUNCH_OK();
  return 0;
}

}  // namespace mdseg
