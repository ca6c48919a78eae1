// mds_bwd.cu — fused backward of  project -> bilinear upsample (align_corners=True) -> OHEM CE
// (SURVEY §8 row a9) in ONE pass: softmax recompute, adjoint of the interpolation and the
// broadcast through G^T, written straight into dlogits_uni.
//
// Reference work replaced (autograd replay of lib/loss/loss_cross_datasets.py:1006-1007 +
// lib/loss/ohem_ce_loss.py:61-90): log_softmax_backward over [B_i,C_ds,H,W], upsample_bilinear2d
// backward (scatter), the einsum backward (bmm) and the index_put into [ΣB,C_uni,h,w].
//
// Work decomposition — one WARP per unit = (image b, class group of 16 dataset classes, strip of low-res columns,
// segment of `seg_rows` cell-rows); a cell-row g interpolates between low-res rows g, g+1.  Two layouts (template ROW):
//   ROW  (w % 32 == 0, w <= 512): the CTA is the w / 32 warps of a row segment, warp i owns columns 32i .. 32i+31 and
//        lane l owns cell x = 32i + l AND column x; the right-column sums of lane 31 reach lane 0 of the next warp
//        through a two-slot shared-memory exchange guarded by full / empty mbarriers (see Lay<ROW> and cell_row);
//   !ROW (any other width): the CTA is one warp owning 28 columns; lane l <= 28 owns cell x = 28*strip + l - 1 (lane 0
//        is the left halo cell, recomputed) and, for l >= 1, column x; nothing is shared between warps.
//   In both the strip width is a multiple of four columns so that finished rows leave as 16-byte stores.
//   * the class planes of rows (g, g+1) arrive as 4-D TMA boxes [8 classes][2 rows][36 cols]
//     in a 2-stage mbarrier ring (lane 0 issues, nobody copies);
//   * per (pixel, class): w*softmax = ex2(z*log2e + (log2 w - lse2)), with the 4..5 x 4..5 label pixels
//     of the cell in registers and the arithmetic packed two columns per instruction (FFMA2/FADD2);
//     per class the cell reduces to 4 sums (upper/lower row x own/right column); the right-column
//     part moves one lane up by shuffle;
//   * the -w*[c == label] term is one packed fp16 compare and two predicated adds per pixel pair;
//   * vertical: the lower-row sums of cell-row g are carried in shared memory and added to the
//     upper-row sums of cell-row g+1, so every low-res row inside a segment is final when it
//     leaves the warp and is broadcast to the unified channels of its class (CSR walk of G, or the
//     identity for the aux heads): the rows of a chunk of classes are parked in a shared-memory tile and
//     written out four (class, channel) pairs per instruction, eight lanes x 16 bytes each.  Only the first row of a segment is incomplete: its two halves
//     go to a scratch plane and a small fix-up kernel adds and broadcasts them.
// Every operand order is fixed, there are no atomics: the gradient is bit-reproducible.
#include "tma_util.cuh"

namespace mdseg {
namespace {

using namespace tma;

constexpr int kKC = 8;                          // classes per TMA stage
constexpr int kBoxW = 36;                       // staged columns: <= 3 alignment + 33
constexpr int kStages = 2;
constexpr int kStageFloats = kKC * 2 * kBoxW;   // 576
constexpr int kStageBytes = kStageFloats * 4;   // 2304
constexpr int kCG = 16;                         // classes per unit
constexpr int kOwn28 = 28;                      // one-warp CTAs: owned columns per strip, 7 aligned groups of four (16-byte stores)
constexpr int kOwn = kOwn28;
constexpr int kStgW28 = 160;                    // one-warp CTAs: staged label columns, <= 15 alignment + 29 cells x 5
constexpr int kMaxR = 5;
constexpr int kEnt = 384;                       // (class, output channel) pairs of one class group cached in shared memory
constexpr uint32_t kNoEnt = 0xffffffffu;

// Shared-memory carve-up of ONE warp.  ROW = false: a CTA is one warp owning 28 columns (lane 0 recomputes the halo cell
// of the strip on its left).  ROW = true: a CTA is the w / 32 warps of a whole low-res row, every lane owns a cell AND a
// column, and the right-column sums of lane 31 travel to lane 0 of the next warp through `xchg` (two slots of
// [kKC classes][upper, lower], guarded by a full / empty mbarrier pair each, in the producer's region).
template <bool ROW>
struct Lay {
  static constexpr int kOwn = ROW ? 32 : kOwn28;
  static constexpr int kStgW = ROW ? 176 : kStgW28;  // ROW: <= 15 alignment + 32 cells x 5
  static constexpr size_t kOffCarry = (size_t)kStages * kStageBytes;
  static constexpr size_t kOffLw = kOffCarry + (size_t)kCG * 32 * 4;
  static constexpr size_t kOffLab = kOffLw + (size_t)kMaxR * kStgW * 4;
  static constexpr size_t kOffEnt = kOffLab + (size_t)kMaxR * kStgW;
  static constexpr size_t kOffTile = kOffEnt + (size_t)kEnt * 4;
  static constexpr size_t kOffEptr = kOffTile + (size_t)kKC * kOwn * 4;
  static constexpr size_t kOffBars = kOffEptr + 16;
  static constexpr size_t kOffXbar = kOffBars + (kStages + 1) * 8;        // ROW: full[2], empty[2]
  static constexpr size_t kOffXchg = kOffXbar + 4 * 8;                    // ROW: [2 slots][kKC][2] floats
  static constexpr size_t kOffC5 = (kOffXchg + 2 * kKC * 2 * 4 + 15) / 16 * 16;        // ROW: [kStages][kKC] float2 fifth-column sums
  static constexpr size_t kSmem = ROW ? ((kOffC5 + (size_t)kStages * kKC * 8 + 127) / 128) * 128 : kOffXbar;
  static_assert(kCG / kKC + 1 <= 4, "eptr holds one quad offset per chunk of a class group, plus the end");
  static_assert(kOffLw % 16 == 0 && kOffLab % 16 == 0 && kOffEnt % 16 == 0 && kOffTile % 16 == 0 && kOffBars % 8 == 0 &&
                    kOffC5 % 16 == 0,
                "shared memory carve-up alignment");
};
static_assert(Lay<false>::kSmem <= 13568, "16 resident one-warp CTAs per SM need <= 13568 bytes of shared memory each");
static_assert(16 * Lay<true>::kSmem <= 232448, "a 16-warp row CTA must fit the 227 KB of one SM");
constexpr size_t kSmem = Lay<false>::kSmem;
constexpr int kMaxRowWarps = 16;

struct GraphDev {
  const int* csr_ptr;  // NULL: identity (output channel = class)
  const int* csr_col;
  const float* csr_val;
  const int* csc_ptr;
  const int* csr4_ptr;  // optional: rows padded to multiples of 4 entries (last entry repeated), in quads
  const int* csr4_col;
};

struct Args {
  mdseg_src_table src;
  const int32_t* dataset_ids;
  const void* labels;
  Geom gm;
  int ignore;
  const float* loss_px;
  const float* lse_px;
  const mdseg_ohem_state* states;
  const float* grad_out;
  float grad_scale;
  void* out_base[MDSEG_MAX_DATASETS];
  long long out_image_stride[MDSEG_MAX_DATASETS];
  int out_channels[MDSEG_MAX_DATASETS];
  GraphDev g[MDSEG_MAX_DATASETS];
  int zero_invalid;  // images with an out-of-range dataset id get zeros in out_base[0]
  float* scrA;       // [n_images][n_seg][c_scr][w]: upper-row half of the first row of a segment
  float* scrB;       // same shape: lower-row half left over by the segment above
  uint8_t* sel8;     // [n_images*H*W]: class of the pixel, 255 = no gradient
  unsigned lite_mask;                  // row CTAs: strips (warps) whose fifth column comes from col5 (host's pick)
  unsigned char lite_strip[kMaxRowWarps];  // the same strips as a list, n_lite long
  int n_lite;
  int c5s;           // class stride of col5: c_scr rounded up to whole chunks (16-byte aligned bulk copies)
  float2* col5;      // row CTAs: [n_images][h-1][w/32][c5s] fifth-column sums (cu, t1) of a strip's one 5-column cell
  int c_scr;
  int seg_rows, n_seg, n_strips;
};

// predicated 8-byte shared-memory store (one instruction; an `if` costs a divergent branch around the address code)
__device__ __forceinline__ void sts2_if(uint32_t on, uint32_t addr, float a, float b) {
  asm volatile("{ .reg .pred q;\n  setp.ne.u32 q, %0, 0;\n  @q st.shared.v2.f32 [%1], {%2, %3}; }"
               :: "r"(on), "r"(addr), "f"(a), "f"(b) : "memory");
}

// e -= |w| where the pixel's class (fp16 pair `lab2`) equals the current class (`c2`): one packed compare, two
// predicated adds.  e holds |w|*softmax, so e - |w|*[c == label] is |w| * d loss / d z.
__device__ __forceinline__ void sub_onehot2(float2& e, uint32_t lab2, uint32_t c2, float nwabs) {
  asm("{ .reg .pred p, q;\n"
      "  setp.eq.f16x2 p|q, %2, %3;\n"
      "  @p add.f32 %0, %0, %4;\n"
      "  @q add.f32 %1, %1, %4; }"
      : "+f"(e.x), "+f"(e.y)
      : "r"(lab2), "r"(c2), "f"(nwabs));
}

// ---- pass 0: selection state of every label pixel in the form the main kernel consumes: the class byte of the
// pixels with a gradient, 255 for the others (the exponent offset log2|w| - lse * log2e is formed by the main kernel
// from the forward's lse rows).  16 pixels per thread and round: four 16-byte loss loads, one 16-byte label load for
// uint8 labels, one 16-byte store.
template <typename L>
__global__ void __launch_bounds__(256) mds_bwd_prep_kernel(const Args a, int64_t px_per_image) {
  const int b = blockIdx.y;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  const bool valid_ds = d >= 0 && d < a.src.n_datasets;
  const int C = valid_ds ? a.src.C[d] : 0;
  SelParams sp;
  sp.thresh = 0.f; sp.kth = 0.f; sp.mode = 0; sp.w = 0.f;
  if (valid_ds) {
    const mdseg_ohem_state* st = a.states + (a.src.seg_per_dataset ? d : 0);
    sp.thresh = st->thresh; sp.kth = st->kth; sp.mode = st->mode;
    sp.w = (a.grad_out ? a.grad_out[a.src.seg_per_dataset ? d : 0] : 1.f) * a.grad_scale * st->inv_n_sel;
  }
  const bool any = valid_ds && fabsf(sp.w) > 0.f;
  const L* labels = (const L*)a.labels;
  const bool lab16 = ((uintptr_t)a.labels & 15) == 0;
  const int64_t base = (int64_t)b * px_per_image;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < px_per_image / 16;
       q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = base + q * 16;
    float4 ls[4];
#pragma unroll
    for (int v = 0; v < 4; ++v) ls[v] = __ldcs(reinterpret_cast<const float4*>(a.loss_px + p) + v);
    uint32_t lab[16];
    if (sizeof(L) == 1 && lab16) {
      const uint4 lv = *reinterpret_cast<const uint4*>((const uint8_t*)a.labels + p);
      const uint32_t wv[4] = {lv.x, lv.y, lv.z, lv.w};
#pragma unroll
      for (int i = 0; i < 16; ++i) lab[i] = (wv[i >> 2] >> (8 * (i & 3))) & 0xffu;
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) lab[i] = (uint32_t)load_label<L>(labels, p + i);
    }
    uint32_t out[4];
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const float lsv[4] = {ls[v].x, ls[v].y, ls[v].z, ls[v].w};
      uint32_t packed = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t lv = lab[4 * v + i];
        const bool sel = any && (lv != (uint32_t)a.ignore) && (lv < (uint32_t)C) && is_selected(sp, lsv[i]);
        packed |= (sel ? lv : 255u) << (8 * i);
      }
      out[v] = packed;
    }
    *reinterpret_cast<uint4*>(a.sel8 + p) = make_uint4(out[0], out[1], out[2], out[3]);
  }
}

// zero rows [r0, r1) (and row h-1 when `last`) of channel u at column x
template <typename TO>
__device__ __forceinline__ void zero_rows(const Args& a, TO* outb, int u, int r0, int r1, bool last, int x, bool own) {
  if (!own) return;
  const int h = a.gm.h, w = a.gm.w;
  for (int r = r0; r < r1; ++r) outb[((int64_t)u * h + r) * w + x] = from_f32<TO>(0.f);
  if (last) outb[((int64_t)u * h + (h - 1)) * w + x] = from_f32<TO>(0.f);
}

struct Unit {
  int lane, b, seg, x, x0, ncols, xl, sx, nx, c_beg, c_end, n_ch, g0, g1, box_x, n_loads, Xa, wst;
  bool own, cached;
  float w_signed, wsign, log2w;
  const float2* c5base;  // lite warps: fifth-column sums of (image, strip, class group) at cell-row 0, else NULL
  int64_t c5row;         // ... and their stride per cell-row
  bool has5;             // this lane owns the five-column cell
};

// four consecutive elements of a gradient row
__device__ __forceinline__ void store4(float* p, const float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void store4(__nv_bfloat16* p, const float4 v) {
  const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
  *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
}
__device__ __forceinline__ void store4(__half* p, const float4 v) {
  const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
  *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
}

// Finished rows of one chunk of classes (tile[class in chunk][column in strip]) -> every output channel of
// those classes.  ents[4q + o] = channel | class-in-chunk << 16 (kNoEnt pads a chunk to whole quads); lane
// octet o takes entry 4q + o, lane t of the octet the columns 4t .. 4t+3 of the strip.
template <typename TO, int OWN>
__device__ __forceinline__ void broadcast_chunk(const Unit& un, TO* orow, const uint32_t* ents, int q0, int q1,
                                                const float* tile, int hw) {
  const int o = un.lane >> 3, t = un.lane & 7;
  const bool col_ok = 4 * t < un.ncols;
  TO* base = orow + 4 * t;
  asm volatile("" : "+l"(base));
  // four quads per round: all entry loads first, then the tile rows, then the stores — the round's shared-memory
  // latencies overlap instead of serialising load -> test -> load -> store four times
  int q = q0;
  for (; q + 4 <= q1; q += 4) {
    uint32_t e[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) e[i] = ents[4 * (q + i) + o];
    float4 v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = *reinterpret_cast<const float4*>(tile + ((e[i] >> 16) & 7u) * OWN + 4 * t);
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (col_ok && e[i] != kNoEnt) store4(base + (int64_t)((e[i] & 0xffffu) * (uint32_t)hw), v[i]);
  }
  for (; q < q1; ++q) {
    const uint32_t e = ents[4 * q + o];
    if (col_ok && e != kNoEnt) {
      const float4 v = *reinterpret_cast<const float4*>(tile + (e >> 16) * OWN + 4 * t);
      store4(base + (int64_t)((e & 0xffffu) * (uint32_t)hw), v);
    }
  }
  __syncwarp();
}

// value v of class group-relative index cg at (row, x): broadcast to the output channels of the class, one
// 4-byte store per channel (fallback for class groups whose channel list does not fit in shared memory)
template <typename TO>
__device__ __forceinline__ void store_class(const Args& a, const GraphDev& gd, const Unit& un, TO* outb, int cg, int row,
                                            float v) {
  const int w = a.gm.w;
  if (gd.csr_ptr == nullptr) {
    if (un.own) outb[((int64_t)(un.c_beg + cg) * a.gm.h + row) * w + un.x] = from_f32<TO>(v);
    return;
  }
  const int e0 = __ldg(gd.csr_ptr + un.c_beg + cg), e1 = __ldg(gd.csr_ptr + un.c_beg + cg + 1);
  for (int e = e0; e < e1; ++e) {
    const int u = __ldg(gd.csr_col + e);
    const float val = gd.csr_val ? __ldg(gd.csr_val + e) : 1.f;
    if (un.own) outb[((int64_t)u * a.gm.h + row) * w + un.x] = from_f32<TO>(v * val);
  }
}

// lane 0: queue the selection state (lse + class byte rows) of cell-row g into shared memory
template <int STGW>
__device__ __forceinline__ void issue_staging(const Args& a, const Unit& un, int Ys, int R, float* lw2s, uint8_t* labs,
                                              uint64_t* sbar) {
  mbar_expect_tx(sbar, (uint32_t)(R * un.wst * 5));
  for (int j = 0; j < R; ++j) {
    const int64_t p = ((int64_t)un.b * a.gm.H + (Ys + j)) * a.gm.W + un.Xa;
    bulk_g2s(lw2s + j * STGW, a.lse_px + p, (uint32_t)(un.wst * 4), sbar);
    bulk_g2s(labs + j * STGW, a.sel8 + p, (uint32_t)un.wst, sbar);
  }
}

// A chunk of a cell-row in which no pixel of the warp is selected: every sum is zero, the finished rows are the
// carried lower-row sums.  Kept out of line so that the hot class loop keeps its registers and code layout.
template <bool ROW>
__device__ __noinline__ void skip_chunk(int lane, int k, int cc, bool own, float* scr_first, int64_t scr_stride,
                                        float* carry, float* tile, float* xslot) {
  constexpr int kOwn = Lay<ROW>::kOwn;
  for (int c = 0; c < cc; ++c) {
    if (ROW && xslot != nullptr && lane == 31) { xslot[2 * c] = 0.f; xslot[2 * c + 1] = 0.f; }
    float* cq = carry + (k * kKC + c) * 32 + lane;
    const float rowv = *cq;
    *cq = 0.f;
    if (scr_first != nullptr) {  // first row of a segment: its upper-row half goes to the scratch plane
      if (own) scr_first[c * scr_stride] = 0.f;
    } else if (ROW) {
      tile[c * kOwn + lane] = rowv;
    } else if (lane >= 1 && lane <= kOwn) {
      tile[c * kOwn + lane - 1] = rowv;
    }
  }
}

// One cell-row: all class chunks of the unit.  RT rows / 4 (+1 when NX5) columns are the compiled loop bounds.
// ROW: `xmine` / `xbar_mine` are this warp's exchange slots and their full[2] / empty[2] barriers (it is the producer for
// the warp on its right), `xleft` / `xbar_left` those of the warp on its left (NULL for the first warp of the row).
// NX5: some cell of the warp has a fifth pixel column, computed in the class loop (scalar tail).  Row CTAs with exactly
// one such lane take NX5 = false with `lite`: the sums of that column come precomputed from mds_bwd_col5_kernel (`c5`:
// the entries of this cell-row's classes, NULL for the other lanes).  A warp with a scalar tail runs ~16 % longer per
// class than its neighbours, the seam exchange makes the whole row CTA wait for it, and a second instantiation of this
// function among the warps of one CTA costs instruction-cache misses on top — so the lite warps run the SAME code.
template <typename TO, int RT, bool NX5, bool ROW>
__device__ __forceinline__ void cell_row(const Args& a, const CUtensorMap* map, const GraphDev& gd, const Unit& un,
                                         TO* outb, int g, int R, int Ys_next, int R_next, const float (&l1w)[5],
                                         const float (&l1h)[kMaxR],
                                         float* stages, uint64_t* bars, float* carry, float* lw2s,
                                         uint8_t* labs, const uint32_t* ents, const int* eptr, float* tile,
                                         float* xmine, uint64_t* xbar_mine, const float* xleft, uint64_t* xbar_left,
                                         bool lite, const float2* c5sm) {
  constexpr int kOwn = Lay<ROW>::kOwn, kStgW = Lay<ROW>::kStgW;
  const int lane = un.lane;
  const float kInf = __int_as_float(0x7f800000);
  // per-pixel exponent offsets and class bytes of this lane's cell, from the staged rows
  float2 LW[RT][2];
  float lw4[RT];
  uint32_t LH[RT][2], lh4[RT];  // class ids as fp16 pairs (255.0 = no gradient), compared two at a time
  uint32_t anysel = 0;          // some pixel of this lane's cell carries a gradient
#pragma unroll
  for (int j = 0; j < RT; ++j) {
    float t[5];
    uint32_t hv[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      t[i] = -kInf;
      hv[i] = 255u;
      if (j < R && i < un.nx) {
        hv[i] = labs[j * kStgW + un.sx + i];
        const float off2 = fmaf(-lw2s[j * kStgW + un.sx + i], kLog2e, un.log2w);  // staged: the forward's lse
        t[i] = hv[i] != 255u ? off2 : -kInf;
      }
      hv[i] = (uint32_t)__half_as_ushort(__ushort2half_rn((unsigned short)hv[i]));
    }
    LW[j][0] = make_float2(t[0], t[1]);
    LW[j][1] = make_float2(t[2], t[3]);
    lw4[j] = t[4];
    LH[j][0] = hv[0] | (hv[1] << 16);
    LH[j][1] = hv[2] | (hv[3] << 16);
    lh4[j] = hv[4] | (0x5bf8u << 16);  // high half 255.0: never a class
    anysel |= (LH[j][0] ^ 0x5bf85bf8u) | (LH[j][1] ^ 0x5bf85bf8u) | (lh4[j] ^ 0x5bf85bf8u);
  }
  __syncwarp();
  if (lane == 0 && g + 1 < un.g1) issue_staging<kStgW>(a, un, Ys_next, R_next, lw2s, labs, &bars[kStages]);
  // No pixel of the warp's 32 cells is selected (OHEM keeps the hard pixels, and those cluster): every term of this
  // cell-row is exactly zero, and the class loops shrink to moving the carried lower-row sums into the finished rows.
  const bool skip = (ROW || un.cached) && !__any_sync(0xffffffffu, anysel != 0);

  float2 L1H[RT];
#pragma unroll
  for (int j = 0; j < RT; ++j) L1H[j] = dup2(l1h[j]);
  const float2 L1W[2] = {make_float2(l1w[0], l1w[1]), make_float2(l1w[2], l1w[3])};
  const float l1w4 = l1w[4];
  const bool first_partial = (g == un.g0) && (un.g0 > 0);
  // first column of the strip in row g of channel 0
  TO* orow = outb + (int64_t)g * a.gm.w + un.x0;
  const float nwabs = -fabsf(un.w_signed);
  const float2 K2 = dup2(kLog2e);  // natural-log logits -> base-2 exponent, folded into the offset FMA

#pragma unroll 1
  for (int k = 0; k < un.n_ch; ++k) {
    const int q = (g - un.g0) * un.n_ch + k;
    const int slot = q % kStages;
    const int c_lo = un.c_beg + k * kKC;
    const int cc = (un.c_end - c_lo) < kKC ? (un.c_end - c_lo) : kKC;

    mbar_wait(&bars[slot], (uint32_t)((q / kStages) & 1));
    const int xs = q & 1;  // exchange slot of this chunk
    if (ROW && xmine != nullptr && q >= 2) mbar_wait(&xbar_mine[2 + xs], (uint32_t)(((q >> 1) - 1) & 1));
    const float* Sp = stages + slot * kStageFloats + un.xl;
    if (skip) {  // warp-uniform
      skip_chunk<ROW>(lane, k, cc, un.own,
                      first_partial ? a.scrA + (((int64_t)un.b * a.n_seg + un.seg) * a.c_scr + c_lo) * a.gm.w + un.x
                                    : nullptr,
                      a.gm.w, carry, tile, xmine ? xmine + xs * kKC * 2 : nullptr);
    } else {
    // corners of the next class are fetched while the current one is being computed (the loop stays rolled)
    float n00 = Sp[0], n01 = Sp[1], n10 = Sp[kBoxW], n11 = Sp[kBoxW + 1];
    uint32_t c2 = class_pair(c_lo);
    // running shared-memory addresses of the class epilogue (re-derived from c they cost ~15 instructions per class)
    float* cp = carry + k * kKC * 32 + lane;
    float* tp = tile + (ROW ? lane : lane - 1);
    uint32_t xaddr = 0, xprod = 0;  // ROW: lane 31 parks its right-column sums for the warp on the right
    if (ROW && xmine != nullptr && lane == 31) { xaddr = smem_u32(xmine + xs * kKC * 2); xprod = 1; }
    asm volatile("" : "+r"(xaddr), "+r"(xprod));
    const float2* x5p = c5sm + slot * kKC;  // lite: this chunk's fifth-column sums arrived with the class planes
#pragma unroll 1
    for (int c = 0; c < cc; ++c, c2 = next_class2(c2)) {
      float v00 = n00, v01 = n01, v10 = n10, v11 = n11;
      Sp += 2 * kBoxW;
      if (c + 1 < cc) { n00 = Sp[0]; n01 = Sp[1]; n10 = Sp[kBoxW]; n11 = Sp[kBoxW + 1]; }
      float2 x5 = make_float2(0.f, 0.f);
      if (!NX5 && un.has5) x5 = x5p[c];
      const float dv0 = v01 - v00, dv1 = v11 - v10;
      const float2 V0 = dup2(v00), DV0 = dup2(dv0), V1 = dup2(v10), DV1 = dup2(dv1);
      float2 CU2, UR2, CL2, LR2;
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        const float2 h0 = fma2(L1W[p], DV0, V0);
        const float2 dd = sub2(fma2(L1W[p], DV1, V1), h0);
        float2 t0, t1;  // first terms assigned, not added to zero (x + 0 is not a no-op the compiler may drop)
#pragma unroll
        for (int j = 0; j < RT; ++j) {
          float2 e = ex2_2(fma2(fma2(L1H[j], dd, h0), K2, LW[j][p]));
          sub_onehot2(e, LH[j][p], c2, nwabs);
          t0 = j == 0 ? e : add2(t0, e);
          t1 = j == 0 ? mul2(L1H[j], e) : fma2(L1H[j], e, t1);
        }
        const float2 cu = sub2(t0, t1);
        CU2 = p == 0 ? cu : add2(CU2, cu);
        UR2 = p == 0 ? mul2(L1W[p], cu) : fma2(L1W[p], cu, UR2);
        CL2 = p == 0 ? t1 : add2(CL2, t1);
        LR2 = p == 0 ? mul2(L1W[p], t1) : fma2(L1W[p], t1, LR2);
      }
      float CU = CU2.x + CU2.y, ur = UR2.x + UR2.y, CL = CL2.x + CL2.y, lr = LR2.x + LR2.y;
      if (!NX5 && lite) {  // warp-uniform; (0, 0) and l1w4 == 0 for the lanes without a fifth column
        CU += x5.x; ur = fmaf(l1w4, x5.x, ur);
        CL += x5.y; lr = fmaf(l1w4, x5.y, lr);
      }
      if (NX5) {
        const float h0 = fmaf(l1w4, dv0, v00);
        const float dd = fmaf(l1w4, dv1, v10) - h0;
        float t0 = 0.f, t1 = 0.f;
#pragma unroll
        for (int j = 0; j < RT; ++j) {
          float2 e = make_float2(ex2_approx(fmaf(fmaf(l1h[j], dd, h0), kLog2e, lw4[j])), 0.f);
          sub_onehot2(e, lh4[j], c2, nwabs);
          t0 += e.x;
          t1 = fmaf(l1h[j], e.x, t1);
        }
        const float cu = t0 - t1;
        CU += cu; ur = fmaf(l1w4, cu, ur);
        CL += t1; lr = fmaf(l1w4, t1, lr);
      }
      const float uo = (CU - ur) * un.wsign;
      const float lo = (CL - lr) * un.wsign;
      ur *= un.wsign;
      lr *= un.wsign;
      float gu = __shfl_up_sync(0xffffffffu, ur, 1);
      float gl = __shfl_up_sync(0xffffffffu, lr, 1);
      if (lane == 0) { gu = 0.f; gl = 0.f; }  // ROW: the left warp's part is added after the class loop
      if (ROW) {
        sts2_if(xprod, xaddr, ur, lr);
        xaddr += 8;
      }
      // vertical: add the lower-row half carried from the cell-row above; the finished row leaves the warp
      const int cg = k * kKC + c;
      const float up = uo + gu;
      const float rowv = up + *cp;
      *cp = lo + gl;
      cp += 32;
      if (first_partial) {
        if (un.own) a.scrA[(((int64_t)un.b * a.n_seg + un.seg) * a.c_scr + (c_lo + c)) * a.gm.w + un.x] = up;
      } else if (ROW || un.cached) {  // row CTAs always cache their channel list (row_route)
        if (ROW || (lane >= 1 && lane <= kOwn)) *tp = rowv;
      } else {
        store_class<TO>(a, gd, un, outb, cg, g, rowv);
      }
      tp += kOwn;
    }
    }  // !skip
    if (ROW) {
      if (xmine != nullptr && lane == 31) mbar_arrive(&xbar_mine[xs]);  // release: the slot is full
      if (xleft != nullptr) {
        // column x0 also receives the right-column sums of the last cell of the warp on the left: lane c adds those of
        // class c to the finished row (or to the scratch half of a segment's first row) and to the carry
        mbar_wait(&xbar_left[xs], (uint32_t)((q >> 1) & 1));
        __syncwarp();
        if (lane < cc) {
          const float xu = xleft[(xs * kKC + lane) * 2], xl = xleft[(xs * kKC + lane) * 2 + 1];
          if (first_partial) {
            a.scrA[(((int64_t)un.b * a.n_seg + un.seg) * a.c_scr + (c_lo + lane)) * a.gm.w + un.x0] += xu;
          } else {
            tile[lane * kOwn] += xu;
          }
          carry[(k * kKC + lane) * 32] += xl;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&xbar_left[2 + xs]);  // the slot may be refilled
      }
    }
    __syncwarp();
    if (lane == 0 && q + kStages < un.n_loads) {  // the slot is free: every lane has read its corners
      const int qn = q + kStages;
      // a class group is one or two chunks (kCG == 2 kKC): no integer division
      const int qrow = un.n_ch == 2 ? qn >> 1 : qn, qk = un.n_ch == 2 ? qn & 1 : 0;
      mbar_expect_tx(&bars[slot], kStageBytes + (un.c5base ? kKC * 8 : 0));
      load_4d(stages + slot * kStageFloats, map, &bars[slot], un.box_x, un.g0 + qrow, un.c_beg + qk * kKC, un.b);
      if (un.c5base)
        bulk_g2s(const_cast<float2*>(c5sm) + slot * kKC, un.c5base + (un.g0 + qrow) * un.c5row + qk * kKC, kKC * 8,
                 &bars[slot]);
    }
    if (un.cached && !first_partial) broadcast_chunk<TO, kOwn>(un, orow, ents, eptr[k], eptr[k + 1], tile, a.gm.h * a.gm.w);
  }
}

template <typename TO, bool ROW>
__global__ void __launch_bounds__(ROW ? 32 * kMaxRowWarps : 32, ROW ? 1 : 16)
mds_bwd_kernel(const __grid_constant__ Maps maps, const __grid_constant__ Args a) {
  using L = Lay<ROW>;
  constexpr int kOwn = L::kOwn, kStgW = L::kStgW;
  extern __shared__ __align__(128) unsigned char smem_all[];
  const int wi = ROW ? (int)(threadIdx.x >> 5) : 0;           // warp of the row CTA = strip
  const int n_w = ROW ? (int)(blockDim.x >> 5) : 1;
  unsigned char* smem_raw = smem_all + (size_t)wi * L::kSmem;
  float* stages = reinterpret_cast<float*>(smem_raw);
  float* carry = reinterpret_cast<float*>(smem_raw + L::kOffCarry); // [kCG][32]
  float* lw2s = reinterpret_cast<float*>(smem_raw + L::kOffLw);     // [kMaxR][kStgW]
  uint8_t* labs = smem_raw + L::kOffLab;                            // [kMaxR][kStgW]
  uint32_t* ents = reinterpret_cast<uint32_t*>(smem_raw + L::kOffEnt);  // [kEnt] channel | class-in-chunk << 16
  float* tile = reinterpret_cast<float*>(smem_raw + L::kOffTile);   // [kKC][kOwn] finished rows of one chunk
  int* eptr = reinterpret_cast<int*>(smem_raw + L::kOffEptr);       // [n_ch + 1] first quad of every chunk
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + L::kOffBars);  // stage ring + staging barrier
  float2* c5sm = reinterpret_cast<float2*>(smem_raw + (ROW ? L::kOffC5 : 0));  // ROW: [kStages][kKC]
  // ROW: exchange with the neighbouring warps (this warp produces for the one on its right)
  const bool has_right = ROW && wi + 1 < n_w, has_left = ROW && wi > 0;
  uint64_t* xbar_mine = has_right ? reinterpret_cast<uint64_t*>(smem_raw + L::kOffXbar) : nullptr;
  float* xmine = has_right ? reinterpret_cast<float*>(smem_raw + L::kOffXchg) : nullptr;
  uint64_t* xbar_left = has_left ? reinterpret_cast<uint64_t*>(smem_raw - L::kSmem + L::kOffXbar) : nullptr;
  const float* xleft = has_left ? reinterpret_cast<const float*>(smem_raw - L::kSmem + L::kOffXchg) : nullptr;

  const Geom& gm = a.gm;
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.z, grp = blockIdx.y;
  const int strip = ROW ? wi : (int)(blockIdx.x % a.n_strips), seg = ROW ? (int)blockIdx.x : (int)(blockIdx.x / a.n_strips);
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  const int h = gm.h, w = gm.w;
  const int x0 = strip * kOwn;
  const int x = ROW ? x0 + lane : x0 + lane - 1;  // ROW: lane l owns cell x0 + l and column x0 + l
  const bool own = ROW ? x <= w - 1 : (lane >= 1 && lane <= kOwn && x <= w - 1);
  const int g0 = seg * a.seg_rows;
  const int g1 = (g0 + a.seg_rows < h - 1) ? g0 + a.seg_rows : h - 1;
  const bool last_seg = (g1 == h - 1);

  if (d < 0 || d >= a.src.n_datasets) {
    if (a.zero_invalid && grp == 0) {
      TO* outb = (TO*)a.out_base[0] + (int64_t)b * a.out_image_stride[0];
      for (int u = 0; u < a.out_channels[0]; ++u) zero_rows<TO>(a, outb, u, g0, g1, last_seg, x, own);
    }
    return;
  }
  const int C = a.src.C[d];
  const int c_beg = grp * kCG;
  if (c_beg >= C) return;
  const int c_end = (c_beg + kCG < C) ? c_beg + kCG : C;
  const GraphDev gd = a.g[d];
  TO* outb = (TO*)a.out_base[d] + (int64_t)b * a.out_image_stride[d];
  const mdseg_ohem_state* st = a.states + (a.src.seg_per_dataset ? d : 0);
  const CUtensorMap* map = &maps.m[d];
  const float wsel = (a.grad_out ? a.grad_out[a.src.seg_per_dataset ? d : 0] : 1.f) * a.grad_scale * st->inv_n_sel;

  // horizontal geometry of this lane's cell
  const bool cell_ok = (x >= 0) && (x <= w - 2) && (ROW || lane <= kOwn);
  int Xbeg = 0, Xend = 0;
  if (cell_ok) cell_span(gm.xm, x, gm.W, Xbeg, Xend);
  const int nx = Xend - Xbeg;
  const unsigned cmask = __ballot_sync(0xffffffffu, cell_ok);
  int Xw0 = 0;
  if (cmask) Xw0 = __shfl_sync(0xffffffffu, Xbeg, __ffs(cmask) - 1);
  float l1w[5];
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    int cell;
    l1w[i] = 0.f;
    if (i < nx) axis_cell(gm.xm, Xbeg + i, cell, l1w[i]);
  }
  // fifth pixel columns: none / one lane of a row-CTA warp (sums precomputed, see cell_row) / anything else (class loop)
  const int n5 = __popc(__ballot_sync(0xffffffffu, nx > 4));
  const bool lite = ROW && a.col5 != nullptr && n5 == 1 && ((a.lite_mask >> strip) & 1u);
  const bool nx5 = n5 > 0 && !lite;

  Unit un;
  un.lane = lane; un.b = b; un.seg = seg; un.x = x; un.nx = nx; un.c_beg = c_beg; un.c_end = c_end;
  un.x0 = x0; un.ncols = (w - x0) < kOwn ? (w - x0) : kOwn;
  un.n_ch = (c_end - c_beg + kKC - 1) / kKC;
  un.g0 = g0; un.g1 = g1; un.own = own;
  un.box_x = ROW ? x0 : ((x0 > 0 ? x0 - 1 : 0) & ~3);
  un.xl = cell_ok ? x - un.box_x : 0;
  un.n_loads = (g1 - g0) * un.n_ch;
  un.Xa = Xw0 & ~15;
  un.sx = cell_ok ? Xbeg - un.Xa : 0;
  un.wst = (gm.W - un.Xa) < kStgW ? (gm.W - un.Xa) : kStgW;
  un.w_signed = wsel; un.wsign = wsel < 0.f ? -1.f : 1.f;
  un.log2w = log2f(fabsf(wsel));  // -inf when nothing is selected or the incoming gradient is 0: every term vanishes
  un.cached = false;
  un.has5 = lite && nx > 4;
  un.c5base = nullptr; un.c5row = 0;
  if (lite) {
    un.c5row = (int64_t)(w / 32) * a.c5s;
    un.c5base = a.col5 + ((int64_t)b * (h - 1) * (w / 32) + strip) * a.c5s + c_beg;
  }

  if (lane == 0) {
    prefetch_map(map);
    for (int s = 0; s <= kStages; ++s) mbar_init(&bars[s], 1);
    if (has_right)
      for (int s = 0; s < 4; ++s) mbar_init(&xbar_mine[s], 1);
    mbar_fence_init();
    {
      int Ys0, Ye0;
      cell_span(gm.ym, g0, gm.H, Ys0, Ye0);
      issue_staging<kStgW>(a, un, Ys0, Ye0 - Ys0, lw2s, labs, &bars[kStages]);
    }
    for (int qn = 0; qn < kStages && qn < un.n_loads; ++qn) {
      mbar_expect_tx(&bars[qn], kStageBytes + (un.c5base ? kKC * 8 : 0));
      load_4d(stages + qn * kStageFloats, map, &bars[qn], un.box_x, g0 + qn / un.n_ch, c_beg + (qn % un.n_ch) * kKC,
              b);
      if (un.c5base)
        bulk_g2s(c5sm + qn * kKC, un.c5base + (g0 + qn / un.n_ch) * un.c5row + (qn % un.n_ch) * kKC, kKC * 8, &bars[qn]);
    }
  }
  for (int cg = 0; cg < kCG; ++cg) carry[cg * 32 + lane] = 0.f;
  // (class, output channel) pairs of this class group, chunk by chunk, each chunk padded to whole quads.  The CSR row
  // starts of the group's classes are fetched by lanes 0..16 in one round trip and the channel ids 32 at a time (a
  // class-by-class walk costs two dependent global loads per class, ~30 round trips during which a row CTA — whose
  // warps all start together — leaves the SM idle).
  static_assert(kCG == 2 * kKC, "the channel-list cache is laid out for two chunks per class group");
  if ((gd.csr_ptr == nullptr || gd.csr_val == nullptr) && a.out_channels[d] <= 0xffff &&
      (int64_t)a.out_channels[d] * h * w < 0x7fffffffLL) {
    const int ncls = c_end - c_beg, nc0 = ncls < kKC ? ncls : kKC;
    int myptr = c_beg + lane;  // identity: entry e is class c_beg + e
    if (gd.csr_ptr != nullptr) myptr = lane <= ncls ? __ldg(gd.csr_ptr + c_beg + lane) : 0;
    const int p0 = __shfl_sync(0xffffffffu, myptr, 0);
    const int p8 = __shfl_sync(0xffffffffu, myptr, nc0);
    const int pe = __shfl_sync(0xffffffffu, myptr, ncls);
    const int len0 = p8 - p0, len1 = pe - p8;
    const int base1 = (len0 + 3) & ~3;
    const int total = base1 + ((len1 + 3) & ~3);
    if (lane == 0) {
      eptr[0] = 0;
      eptr[1] = base1 >> 2;
      eptr[un.n_ch] = total >> 2;  // n_ch == 1: len1 == 0 and total == base1
    }
    for (int eb = 0; eb < pe - p0; eb += 32) {
      const int e = eb + lane;
      int cls = 0;  // class of entry e within the group: number of row starts (classes 1..ncls-1) at or below it
#pragma unroll
      for (int j = 1; j < kCG; ++j) {
        const int pj = __shfl_sync(0xffffffffu, myptr, j);
        cls += (j < ncls && pj <= p0 + e) ? 1 : 0;
      }
      if (e < pe - p0) {
        const int u = gd.csr_ptr != nullptr ? __ldg(gd.csr_col + p0 + e) : c_beg + e;
        const int pos = cls < kKC ? e : base1 + (e - len0);
        if (pos < kEnt) ents[pos] = (uint32_t)u | ((uint32_t)(cls & (kKC - 1)) << 16);
      }
    }
    if (lane < base1 - len0 && len0 + lane < kEnt) ents[len0 + lane] = kNoEnt;
    if (lane < total - base1 - len1 && base1 + len1 + lane < kEnt) ents[base1 + len1 + lane] = kNoEnt;
    un.cached = total <= kEnt;
  }
  __syncwarp();
  if (ROW) __syncthreads();  // the neighbours' exchange barriers are initialised (every early exit above is CTA-uniform)

  // label-row range of every cell-row of the segment: lane t holds the first label row of cell-row g0 + t
  int ys_tab = gm.H;
  if (g0 + lane < h - 1) ys_tab = first_dst_ge(gm.ym, g0 + lane, gm.H);
  for (int g = g0; g < g1; ++g) {
    const int Ys = __shfl_sync(0xffffffffu, ys_tab, g - g0);
    const int Ye = __shfl_sync(0xffffffffu, ys_tab, g - g0 + 1);
    const int R = Ye - Ys;
    float l1h[kMaxR];
#pragma unroll
    for (int j = 0; j < kMaxR; ++j) {
      int cell;
      l1h[j] = 0.f;
      if (j < R) axis_cell(gm.ym, Ys + j, cell, l1h[j]);
    }
    const int Rn = __shfl_sync(0xffffffffu, ys_tab, (g - g0 + 2) & 31) - Ye;  // rows of the next cell-row
    mbar_wait(&bars[kStages], (uint32_t)((g - g0) & 1));
#define MDSEG_ROW(RT, N5)                                                                                           \
  cell_row<TO, RT, N5, ROW>(a, map, gd, un, outb, g, R, Ye, Rn, l1w, l1h, stages, bars, carry, lw2s, labs, ents, eptr, \
                            tile, xmine, xbar_mine, xleft, xbar_left, lite, c5sm)
    if (R <= 4) {
      if (nx5) MDSEG_ROW(4, true); else MDSEG_ROW(4, false);
    } else {
      if (nx5) MDSEG_ROW(5, true); else MDSEG_ROW(5, false);
    }
#undef MDSEG_ROW
  }

  // what is left in the carry is the lower-row half of row g1
  if (last_seg && un.cached) {
    TO* olast = outb + (int64_t)(h - 1) * w + x0;
    for (int k = 0; k < un.n_ch; ++k) {
      for (int j = 0; j < kKC && k * kKC + j < c_end - c_beg; ++j)
        if (ROW) tile[j * kOwn + lane] = carry[(k * kKC + j) * 32 + lane];
        else if (lane >= 1 && lane <= kOwn) tile[j * kOwn + lane - 1] = carry[(k * kKC + j) * 32 + lane];
      __syncwarp();
      broadcast_chunk<TO, kOwn>(un, olast, ents, eptr[k], eptr[k + 1], tile, h * w);
    }
  } else {
    for (int cg = 0; cg < c_end - c_beg; ++cg) {
      const float v = carry[cg * 32 + lane];
      if (last_seg) {
        store_class<TO>(a, gd, un, outb, cg, h - 1, v);
      } else if (own) {
        a.scrB[(((int64_t)b * a.n_seg + (seg + 1)) * a.c_scr + (c_beg + cg)) * w + x] = v;
      }
    }
  }
  // unified classes no dataset class maps to: zero gradient
  if (grp == 0 && gd.csr_ptr != nullptr && gd.csc_ptr != nullptr) {
    for (int u0 = 0; u0 < a.out_channels[d]; u0 += 32) {
      const int u = u0 + lane;
      const bool empty = u < a.out_channels[d] && __ldg(gd.csc_ptr + u) == __ldg(gd.csc_ptr + u + 1);
      unsigned m = __ballot_sync(0xffffffffu, empty);
      while (m) {
        const int uu = u0 + __ffs(m) - 1;
        m &= m - 1;
        zero_rows<TO>(a, outb, uu, g0, g1, last_seg, x, own);
      }
    }
  }
}

// Row CTAs: the fifth pixel column of a warp strip's ONE five-column cell, for every class — what cell_row<N5 = 1>
// computes in its scalar tail, in the same operation order (the gradient is bit-identical either way), written as
// (cu, t1) = (upper-row sum, lower-row sum) of that column.  CTA = the candidate strips of cell-row g of image b, one
// warp each; a warp whose strip has no such cell (or several: those stay in the class loop) leaves at once; lanes walk
// the classes.  At stride 4 a row has W - 4 (w - 1) five-column cells (4 of 511 at 2048 -> 512).  The host lists the
// candidate strips (a.lite_strip) only to keep the grid small; whether a strip is taken is decided here and in the main
// kernel by the same device code.
__global__ void __launch_bounds__(32 * kMaxRowWarps) mds_bwd_col5_kernel(const Args a) {
  const Geom& gm = a.gm;
  const int lane = threadIdx.x & 31, strip = a.lite_strip[threadIdx.x >> 5], n_w = a.gm.w / 32;
  const int g = blockIdx.x, b = blockIdx.y;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  if (d < 0 || d >= a.src.n_datasets) return;
  const int h = gm.h, w = gm.w;
  const int x = strip * 32 + lane;
  int Xbeg = 0, Xend = 0;
  if (x <= w - 2) cell_span(gm.xm, x, gm.W, Xbeg, Xend);
  const unsigned m5 = __ballot_sync(0xffffffffu, Xend - Xbeg > 4);
  if (__popc(m5) != 1) return;
  const int owner = __ffs(m5) - 1;
  const int xo = strip * 32 + owner;
  const int X5 = __shfl_sync(0xffffffffu, Xbeg, owner) + 4;
  int cell;
  float l1w4;
  axis_cell(gm.xm, X5, cell, l1w4);
  int Ys, Ye;
  cell_span(gm.ym, g, gm.H, Ys, Ye);
  const int R = Ye - Ys;
  const int C = a.src.C[d];
  const mdseg_ohem_state* st = a.states + (a.src.seg_per_dataset ? d : 0);
  const float wsel = (a.grad_out ? a.grad_out[a.src.seg_per_dataset ? d : 0] : 1.f) * a.grad_scale * st->inv_n_sel;
  const float log2w = log2f(fabsf(wsel)), nwabs = -fabsf(wsel);
  const float kInf = __int_as_float(0x7f800000);
  float l1h[kMaxR], off[kMaxR];
  int cls[kMaxR];
#pragma unroll
  for (int j = 0; j < kMaxR; ++j) {
    l1h[j] = 0.f; off[j] = -kInf; cls[j] = 255;
    if (j < R) {
      axis_cell(gm.ym, Ys + j, cell, l1h[j]);
      const int64_t p = ((int64_t)b * gm.H + (Ys + j)) * gm.W + X5;
      cls[j] = a.sel8[p];
      if (cls[j] != 255) off[j] = fmaf(-a.lse_px[p], kLog2e, log2w);
    }
  }
  const float* yb = (const float*)a.src.base[d] + (int64_t)b * a.src.image_stride[d] + (int64_t)g * w + xo;
  float2* out = a.col5 + ((((int64_t)b * (h - 1) + g) * n_w + strip) * a.c5s);
  for (int c = lane; c < C; c += 32) {
    const float* yc = yb + (int64_t)c * h * w;
    const float v00 = yc[0], v01 = yc[1], v10 = yc[w], v11 = yc[w + 1];
    const float dv0 = v01 - v00, dv1 = v11 - v10;
    const float h0 = fmaf(l1w4, dv0, v00);
    const float dd = fmaf(l1w4, dv1, v10) - h0;
    float t0 = 0.f, t1 = 0.f;
#pragma unroll
    for (int j = 0; j < kMaxR; ++j) {
      if (j < R) {
        float e = ex2_approx(fmaf(fmaf(l1h[j], dd, h0), kLog2e, off[j]));
        if (cls[j] == c) e += nwabs;
        t0 += e;
        t1 = fmaf(l1h[j], e, t1);
      }
    }
    out[c] = make_float2(t0 - t1, t1);
  }
}

// first row of every segment but the first: sum of the two halves, broadcast to the output channels
template <typename TO>
__global__ void __launch_bounds__(256) mds_bwd_fixup_kernel(const Args a) {
  const int b = blockIdx.z, k = blockIdx.y + 1;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  if (d < 0 || d >= a.src.n_datasets) return;
  const int C = a.src.C[d];
  const int w = a.gm.w, h = a.gm.h, w4 = w / 4;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int cls = idx / w4, x4 = idx - cls * w4;
  if (cls >= C) return;
  const int row = k * a.seg_rows;
  const int64_t so = (((int64_t)b * a.n_seg + k) * a.c_scr + cls) * w + x4 * 4;
  const float4 A = *reinterpret_cast<const float4*>(a.scrA + so);
  const float4 B = *reinterpret_cast<const float4*>(a.scrB + so);
  const float v[4] = {A.x + B.x, A.y + B.y, A.z + B.z, A.w + B.w};
  const GraphDev gd = a.g[d];
  TO* outb = (TO*)a.out_base[d] + (int64_t)b * a.out_image_stride[d];
  if (gd.csr_ptr == nullptr) {
    TO* o = outb + ((int64_t)cls * h + row) * w + x4 * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = from_f32<TO>(v[i]);
    return;
  }
  const int e0 = __ldg(gd.csr_ptr + cls), e1 = __ldg(gd.csr_ptr + cls + 1);
  for (int e = e0; e < e1; ++e) {
    const int u = __ldg(gd.csr_col + e);
    const float val = gd.csr_val ? __ldg(gd.csr_val + e) : 1.f;
    TO* o = outb + ((int64_t)u * h + row) * w + x4 * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = from_f32<TO>(v[i] * val);
  }
}

// cell-rows per unit: the per-unit set-up and the seam fix-up are amortised over 16 rows (8 and 30 measured within 3 %)
#ifndef MDSEG_SEG_ROWS
#define MDSEG_SEG_ROWS 16
#endif
// Small batches of row CTAs (cfg1; a few images per rank under strong scaling) would leave most SMs without a CTA at 16
// rows per segment: halve the segment until the grid — segments x class groups of the widest dataset x images, an upper
// bound without reading the dataset ids — reaches one CTA per SM, not below 4 rows (the seam fix-up grows with it).
int pick_seg_rows(int h, int w, int n_images, int c_max) {
  int sr = h - 1 < MDSEG_SEG_ROWS ? h - 1 : MDSEG_SEG_ROWS;
  if (sr < 1) sr = 1;
  if (!(w % 32 == 0 && w / 32 <= kMaxRowWarps)) return sr;
  const long long per_seg = (long long)n_images * ((c_max + kCG - 1) / kCG);
  while (sr > 4 && per_seg * ((h - 1 + sr - 1) / sr) < sm_count()) sr /= 2;
  return sr;
}

template <typename L>
int launch_prep(const Args& a, int n_images, cudaStream_t s) {
  const int64_t ppi = (int64_t)a.gm.H * a.gm.W;
  int64_t bx = ceil_div64(ppi / 16, 256);
  const int64_t want = ceil_div64((int64_t)sm_count() * 16, n_images);
  if (bx > want) bx = want;
  mds_bwd_prep_kernel<L><<<dim3((unsigned)bx, (unsigned)n_images), 256, 0, s>>>(a, ppi);
  MDSEG_LAUNCH_OK();
  return 0;
}

// Row CTAs (one warp per 32 columns, no halo cells, no idle lanes) when the row is a whole number of warps that fit one
// CTA and every class group's channel list fits the shared-memory cache (`ents_fit`: the uncached per-class stores
// cannot take the neighbour's column-0 contribution).
bool row_route(const Args& a, bool ents_fit) {
  return ents_fit && a.gm.w % 32 == 0 && a.gm.w / 32 <= kMaxRowWarps;
}

template <typename TO>
int launch(const char* who, int label_dtype, const Maps& maps, const Args& a, int n_images, int max_c, bool ents_fit,
           cudaStream_t s) {
  if (int rc = with_int_type(label_dtype, who, "label dtype", [&](auto l) {
        return launch_prep<typename decltype(l)::type>(a, n_images, s);
      }))
    return rc;
  if (row_route(a, ents_fit)) {
    const int n_w = a.gm.w / 32;
    if (a.col5 != nullptr && a.n_lite > 0) {
      mds_bwd_col5_kernel<<<dim3((unsigned)(a.gm.h - 1), (unsigned)n_images), 32 * a.n_lite, 0, s>>>(a);
      MDSEG_LAUNCH_OK();
    }
    const size_t smem = (size_t)n_w * Lay<true>::kSmem;
    auto k = mds_bwd_kernel<TO, true>;
    MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((unsigned)a.n_seg, (unsigned)((max_c + kCG - 1) / kCG), (unsigned)n_images);
    k<<<grid, 32 * n_w, smem, s>>>(maps, a);
  } else {
    auto k = mds_bwd_kernel<TO, false>;
    MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem));
    dim3 grid((unsigned)(a.n_strips * a.n_seg), (unsigned)((max_c + kCG - 1) / kCG), (unsigned)n_images);
    k<<<grid, 32, kSmem, s>>>(maps, a);
  }
  MDSEG_LAUNCH_OK();
  if (a.n_seg > 1) {
    dim3 g2((unsigned)(((int64_t)max_c * (a.gm.w / 4) + 255) / 256), (unsigned)(a.n_seg - 1), (unsigned)n_images);
    mds_bwd_fixup_kernel<TO><<<g2, 256, 0, s>>>(a);
    MDSEG_LAUNCH_OK();
  }
  return 0;
}

// fifth-column table of the row CTAs (0 when the width does not take that route)
size_t col5_bytes(int n_images, int h, int w, int c_max) {
  if (w % 32 != 0 || w / 32 > kMaxRowWarps || h < 2) return 0;
  return (size_t)n_images * (h - 1) * (w / 32) * ((c_max + kKC - 1) / kKC * kKC) * sizeof(float2) + 16;
}

// Strips of 32 cells with exactly one five-column cell (host replica of AxisMap::floor_at — one fp32 multiply and a
// truncation, the same on both sides; the kernels re-derive the answer and only use this list to prune work).
void pick_lite_strips(Args& a) {
  a.lite_mask = 0; a.n_lite = 0;
  if (a.col5 == nullptr) return;
  const int w = a.gm.w, W = a.gm.W;
  int n5[kMaxRowWarps] = {0};
  int cols = 0, cur = 0;
  for (int X = 0; X <= W; ++X) {
    int cell = w - 2;
    if (X < W) {
      const int i0 = (int)(a.gm.xm.scale * (float)X);
      cell = i0 > w - 2 ? w - 2 : i0;
    }
    if (X == W || cell != cur) {
      if (cols > 4 && cur / 32 < kMaxRowWarps) ++n5[cur / 32];
      cur = cell; cols = 0;
    }
    ++cols;
  }
  for (int st = 0; st < w / 32 && st < kMaxRowWarps; ++st)
    if (n5[st] == 1) {
      a.lite_mask |= 1u << st;
      a.lite_strip[a.n_lite++] = (unsigned char)st;
    }
}

// The fused kernel covers fp32 sources at up-sampling factors in [1, 5] (tma::fast_geometry) whose label rows are whole
// 16-byte bulk copies.
bool fused_geometry(const mdseg_src_table* src, const Geom& gm) {
  return gm.W % 16 == 0 && tma::fast_geometry(*src, gm);
}

// ... and, behind a projection, column-one-hot sparse graphs
bool fused_route(const mdseg_src_table* src, const mdseg_graph_table* graphs, const Geom& gm) {
  for (int i = 0; i < src->n_datasets; ++i) {
    const mdseg_sparse_graph& g = graphs->g[i];
    if (g.dense || !g.col_onehot || !g.csr_ptr || !g.csc_ptr || g.C_ds != src->C[i]) return false;
  }
  return fused_geometry(src, gm);
}

// the fused kernel's workspace: the two seam halves of every segment, the class byte of every pixel, the fifth columns
size_t fused_workspace_bytes(int n_images, const Geom& gm, int c_max) {
  const int sr = pick_seg_rows(gm.h, gm.w, n_images, c_max);
  const int n_seg = (gm.h - 1 + sr - 1) / sr;
  return 2 * (size_t)n_images * n_seg * c_max * gm.w * 4 + (size_t)n_images * gm.H * gm.W + 1024 +
         col5_bytes(n_images, gm.h, gm.w, c_max);
}

// The Args fields both fused entry points share, the workspace carved into them and the sources' tensor maps; the
// caller adds the output rows, the channel lists and zero_invalid.
int setup_fused(const char* who, const mdseg_src_table* src, const int32_t* dataset_ids, const void* labels,
                const Geom& gm, int n_images, int ignore, const float* loss_px, const float* lse_px,
                mdseg_ohem_state* states, const float* grad_out, float grad_scale, float* ws, Args& a, Maps* maps) {
  MDSEG_REQUIRE(((uintptr_t)loss_px & 15) == 0 && ((uintptr_t)lse_px & 15) == 0,
                "%s: loss_px / lse_px must be 16-byte aligned", who);
  const int c_max = max_c(src), h = gm.h, w = gm.w;
  a.src = *src; a.dataset_ids = dataset_ids; a.labels = labels; a.gm = gm; a.ignore = ignore;
  a.loss_px = loss_px; a.lse_px = lse_px; a.states = states; a.grad_out = grad_out; a.grad_scale = grad_scale;
  a.seg_rows = pick_seg_rows(h, w, n_images, c_max);
  a.n_seg = (h - 1 + a.seg_rows - 1) / a.seg_rows;
  a.n_strips = (w + kOwn - 1) / kOwn;
  a.c_scr = c_max;
  a.scrA = ws;
  a.scrB = ws + (size_t)n_images * a.n_seg * c_max * w;
  a.sel8 = reinterpret_cast<uint8_t*>(a.scrB + (size_t)n_images * a.n_seg * c_max * w);
  a.col5 = col5_bytes(n_images, h, w, c_max)
               ? reinterpret_cast<float2*>(((uintptr_t)(a.sel8 + (size_t)n_images * gm.H * gm.W) + 15) & ~(uintptr_t)15)
               : nullptr;
  a.c5s = (c_max + kKC - 1) / kKC * kKC;
  pick_lite_strips(a);
  return make_maps(a.src, gm, n_images, kBoxW, 2, kKC, maps);
}

}  // namespace
}  // namespace mdseg

extern "C" size_t mdseg_mds_bwd_workspace_bytes(const mdseg_src_table* src, const mdseg_graph_table* graphs,
                                                int n_images, int h, int w, int H, int W) {
  using namespace mdseg;
  if (!src_count_ok(src) || !graphs || graphs->n_datasets != src->n_datasets || n_images <= 0 || h <= 0 || w <= 0 ||
      H <= 0 || W <= 0)
    return 256;
  const int c_max = max_c(src);
  const Geom gm = make_geom(h, w, H, W);
  if (fused_route(src, graphs, gm)) return fused_workspace_bytes(n_images, gm, c_max);
  // generic route: two gradient planes + the converted dense graphs of mdseg_proj_bwd_tc
  return 2 * (size_t)n_images * c_max * h * w * 4 + 512 + mdseg_proj_bwd_tc_workspace_bytes(graphs, MDSEG_F32);
}

extern "C" int mdseg_mds_bwd(const mdseg_src_table* src, const mdseg_graph_table* graphs, const int32_t* dataset_ids,
                             const void* labels, int label_dtype, int n_images, int h, int w, int H, int W, int ignore,
                             const float* loss_px, const float* lse_px, mdseg_ohem_state* states,
                             const float* grad_out, float grad_scale, void* dx, int dx_dtype, void* workspace,
                             size_t workspace_bytes, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(src_count_ok(src) && graph_header_ok(graphs) && graphs->n_datasets == src->n_datasets,
                "mdseg_mds_bwd: bad source / graph table");
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0 && H > 0 && W > 0 && h <= 65535,
                "mdseg_mds_bwd: bad shape");
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(labels && loss_px && lse_px && states && dx && workspace, "mdseg_mds_bwd: null pointer");
  MDSEG_REQUIRE(is_float_dtype(dx_dtype), "mdseg_mds_bwd: unsupported gradient dtype %d", dx_dtype);
  const int c_max = max_c(src);
  MDSEG_REQUIRE(workspace_bytes >= mdseg_mds_bwd_workspace_bytes(src, graphs, n_images, h, w, H, W),
                "mdseg_mds_bwd: workspace too small");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t hw = (int64_t)h * w;
  float* ws = reinterpret_cast<float*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  const Geom gm = make_geom(h, w, H, W);

  if (!fused_route(src, graphs, gm)) {
    // generic route: adjoint of the upsample into two planes, then the projection adjoint
    float* dyA = ws;
    float* dyB = ws + (size_t)n_images * c_max * hw;
    mdseg_src_table dA = *src, dB = *src;
    dA.dtype = MDSEG_F32; dB.dtype = MDSEG_F32; dA.cmax = nullptr; dB.cmax = nullptr;
    for (int i = 0; i < src->n_datasets; ++i) {
      dA.base[i] = dyA; dB.base[i] = dyB;
      dA.image_stride[i] = (long long)c_max * hw; dB.image_stride[i] = (long long)c_max * hw;
      dA.C_alloc[i] = c_max; dB.C_alloc[i] = c_max;
    }
    if (int rc = mdseg_up_ce_bwd(src, dataset_ids, labels, label_dtype, n_images, h, w, H, W, ignore, loss_px, lse_px,
                                 states, grad_out, grad_scale, &dA, &dB, stream))
      return rc;
    // dense graphs: adjoint on the tensor cores, converted graphs behind the two planes in the workspace
    float* tail = dyB + (size_t)n_images * c_max * hw;
    const size_t used = (size_t)((unsigned char*)tail - (unsigned char*)workspace);
    return mdseg_proj_bwd_tc(dyA, dyB, c_max, graphs, dataset_ids, n_images, h, w, dx, dx_dtype, tail,
                             workspace_bytes - used, stream);
  }

  Args a;
  Maps maps;
  if (int rc = setup_fused("mdseg_mds_bwd", src, dataset_ids, labels, gm, n_images, ignore, loss_px, lse_px, states,
                           grad_out, grad_scale, ws, a, &maps))
    return rc;
  for (int i = 0; i < MDSEG_MAX_DATASETS; ++i) {
    a.out_base[i] = dx; a.out_image_stride[i] = (long long)graphs->C_uni * hw; a.out_channels[i] = graphs->C_uni;
    a.g[i] = GraphDev{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    if (i < src->n_datasets) {
      const mdseg_sparse_graph& g = graphs->g[i];
      a.g[i] = GraphDev{g.csr_ptr, g.csr_col, g.csr_val, g.csc_ptr, g.csr4_ptr, g.csr4_col};
    }
  }
  a.zero_invalid = 1;
  bool ents_fit = true;  // a class group's (class, channel) pairs, each chunk padded to quads, within kEnt
  for (int i = 0; i < src->n_datasets; ++i) ents_fit = ents_fit && graphs->g[i].nnz + 8 <= kEnt;
  return with_float_type(dx_dtype, "mdseg_mds_bwd", "gradient dtype", [&](auto t) {
    return launch<typename decltype(t)::type>("mdseg_mds_bwd", label_dtype, maps, a, n_images, c_max, ents_fit, s);
  });
}

// ---- the same kernel without a projection: aux heads (a10) and any direct upsample + CE --------------------
extern "C" size_t mdseg_up_ce_bwd_direct_workspace_bytes(const mdseg_src_table* src, int n_images, int h, int w, int H,
                                                         int W) {
  using namespace mdseg;
  if (!src_count_ok(src) || n_images <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return 256;
  const Geom gm = make_geom(h, w, H, W);
  if (fused_geometry(src, gm)) return fused_workspace_bytes(n_images, gm, max_c(src));
  return two_plane_bytes(src, n_images, h, w);
}

extern "C" int mdseg_up_ce_bwd_direct_is_fused(const mdseg_src_table* src, int h, int w, int H, int W) {
  using namespace mdseg;
  if (!src_count_ok(src) || h <= 0 || w <= 0 || H <= 0 || W <= 0) return 0;
  return fused_geometry(src, make_geom(h, w, H, W)) ? 1 : 0;
}

extern "C" int mdseg_up_ce_bwd_direct(const mdseg_src_table* src, const int32_t* dataset_ids, const void* labels,
                                      int label_dtype, int n_images, int h, int w, int H, int W, int ignore,
                                      const float* loss_px, const float* lse_px, mdseg_ohem_state* states,
                                      const float* grad_out, float grad_scale, const mdseg_src_table* dst,
                                      void* workspace, size_t workspace_bytes, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(src_count_ok(src) && dst && dst->n_datasets == src->n_datasets && is_float_dtype(dst->dtype),
                "mdseg_up_ce_bwd_direct: bad source / destination table");
  for (int i = 0; i < src->n_datasets; ++i)
    MDSEG_REQUIRE(dst->base[i] && dst->C[i] == src->C[i], "mdseg_up_ce_bwd_direct: destination %d does not match", i);
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0 && H > 0 && W > 0 && h <= 65535,
                "mdseg_up_ce_bwd_direct: bad shape");
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(labels && loss_px && lse_px && states && workspace, "mdseg_up_ce_bwd_direct: null pointer");
  MDSEG_REQUIRE(workspace_bytes >= mdseg_up_ce_bwd_direct_workspace_bytes(src, n_images, h, w, H, W),
                "mdseg_up_ce_bwd_direct: workspace too small");
  cudaStream_t s = (cudaStream_t)stream;
  const Geom gm = make_geom(h, w, H, W);

  if (!fused_geometry(src, gm)) {
    // generic route: two planes per dataset (zero for the images of other datasets), then their sum
    return two_plane_adjoint("mdseg_up_ce_bwd_direct", src, dst, n_images, h, w, workspace, true, s,
                             [&](const mdseg_src_table& dA, const mdseg_src_table& dB) {
                               return mdseg_up_ce_bwd(src, dataset_ids, labels, label_dtype, n_images, h, w, H, W,
                                                      ignore, loss_px, lse_px, states, grad_out, grad_scale, &dA, &dB,
                                                      stream);
                             });
  }

  float* ws = reinterpret_cast<float*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  Args a;
  Maps maps;
  if (int rc = setup_fused("mdseg_up_ce_bwd_direct", src, dataset_ids, labels, gm, n_images, ignore, loss_px, lse_px,
                           states, grad_out, grad_scale, ws, a, &maps))
    return rc;
  for (int i = 0; i < MDSEG_MAX_DATASETS; ++i) {
    const bool on = i < src->n_datasets;
    a.out_base[i] = on ? const_cast<void*>(dst->base[i]) : nullptr;
    a.out_image_stride[i] = on ? dst->image_stride[i] : 0;
    a.out_channels[i] = on ? src->C[i] : 0;
    a.g[i] = GraphDev{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // identity: channel = class
  }
  a.zero_invalid = 0;  // rows of images that do not belong to a head stay as the caller initialised them
  const int c_max = max_c(src);
  // identity channel lists: 16 entries per class group
  return with_float_type(dst->dtype, "mdseg_up_ce_bwd_direct", "destination dtype", [&](auto t) {
    return launch<typename decltype(t)::type>("mdseg_up_ce_bwd_direct", label_dtype, maps, a, n_images, c_max, true, s);
  });
}
