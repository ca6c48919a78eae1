// up_ce_tma.cu — TMA-pipelined fused bilinear upsample (align_corners=True) + CE,
// forward and adjoint: the fast path of mdseg_up_ce_fwd / mdseg_up_ce_bwd for fp32
// low-res logits at up-sampling factors <= 5 (the training geometry: stride 4).
// Reference work replaced: lib/loss/loss_cross_datasets.py:1007,1051 +
// lib/loss/ohem_ce_loss.py:27,61 and their autograd replay (see up_ce.cu).
//
// Structure (per CTA = one image, one low-res row g, 128 threads):
//   * the class planes of the two low-res rows (g, g+1) arrive as 4-D TMA boxes
//     [16 classes][2 rows][132 cols] in a 3-stage (fwd) / 2-stage (bwd) mbarrier ring —
//     one elected thread issues cp.async.bulk.tensor, nobody spends issue slots on staging;
//   * thread = one low-res cell; its 4 corners are 4 LDS per class, reused by the
//     4x4 (max 5x5) label pixels of the cell held in registers;
//   * per (pixel, class): 1 FFMA + 1 MUFU.EX2 + 1 FADD.  With hm0/dm = the interpolation
//     of the per-corner channel maxima along x (loop invariant per column i),
//        E_i = h0_i - hm0_i,  D_i = (h1_i - h0_i) - dm_i   (5 ops per column and class)
//        log2e*(z_ji - M_ji) = fma(l1h_j, D_i, E_i)
//     M (bilinear interpolation of the channel maximum) bounds every z from above, so
//     the softmax needs no running maximum;
//   * labels are staged per warp as bytes with coalesced loads; loss / lse leave through
//     a per-warp row buffer as contiguous 4-byte rows;
//   * backward: w*softmax = ex2(z2 - (lse2 - log2 w)) — one FFMA, FADD, MUFU, FADD, FFMA
//     per (pixel, class); per class the cell keeps 4 sums (upper/lower plane x own/right
//     cell); the right-cell part moves one lane up with a shuffle (warps overlap by one
//     cell, so nothing crosses a warp); the -w*[c==label] term is one shared-memory
//     scatter per pixel.  Planes A[g] / B[g+1] are written with plain stores.
#include <cuda.h>
#include <float.h>

#include "tma_util.cuh"

namespace mdseg {
namespace {

constexpr int kT = 128;        // threads per CTA
constexpr int kNW = kT / 32;   // warps
constexpr int kBoxW = 132;     // staged columns per row (528 B, multiple of 16)
constexpr int kKC = 16;        // classes per TMA stage
constexpr int kStageFloats = kKC * 2 * kBoxW;
constexpr int kStageBytes = kStageFloats * 4;  // 16896
constexpr int kFwdStages = 3;
constexpr int kBwdStages = 2;
constexpr int kMaxR = 5, kMaxNX = 5;
constexpr int kRowBuf = 32 * kMaxNX;  // label columns covered by one warp
constexpr int kOwnPerWarp = 31;       // backward: lane 0 of every warp is a halo cell

struct alignas(64) TmaMaps {
  CUtensorMap m[MDSEG_MAX_DATASETS];
};

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "MDSEG_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra MDSEG_DONE;\n"
      "bra MDSEG_WAIT;\n"
      "MDSEG_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// ---- per-warp staging of labels / per-pixel floats -------------------------------------------
// lab_w[j*kRowBuf + k] = label of pixel (Yb+j, Xw0+k) as a byte; 255 = ignored or invalid.
template <typename L>
__device__ __forceinline__ void stage_labels(uint8_t* lab_w, const L* labels, int64_t img_row0, int W, int R, int Xw0,
                                             int nw, int C, int ignore, int& err) {
  const int lane = threadIdx.x & 31;
  for (int j = 0; j < R; ++j) {
    const int64_t base = (img_row0 + j) * W + Xw0;
    for (int k = lane; k < nw; k += 32) {
      const int lab = load_label<L>(labels, base + k);
      uint8_t v = 255;
      if (lab != ignore) {
        if ((unsigned)lab < (unsigned)C) v = (uint8_t)lab;
        else err |= MDSEG_ERR_LABEL_RANGE;
      }
      lab_w[j * kRowBuf + k] = v;
    }
  }
}

struct Stats {
  unsigned n_valid = 0, n_hard = 0, n_px = 0;
  float sum_hard = 0.f;
};

// =================================================================================================
// forward
// =================================================================================================
template <typename L, int R, int NX>
__device__ __forceinline__ void fwd_tile(const FwdArgs& a, const CUtensorMap* map, int C, int b, int g, int Ys, int xa,
                                         int xl, int Xbeg, int nx, int Xw0, int nw, float* stages, uint64_t* bars,
                                         const float* cm, const uint8_t* lab_w, float* rb, float thresh, Stats& st) {
  const Geom& gm = a.gm;
  const int lane = threadIdx.x & 31;
  const int off = Xbeg - Xw0;
  float l1w[NX], hm0[NX], dm[NX], l1h[R];
#pragma unroll
  for (int j = 0; j < R; ++j) {
    int i0, i1;
    float l0;
    gm.ym.at(Ys + j, i0, i1, l0, l1h[j]);
  }
  {
    const float c00 = cm[xl], c01 = cm[xl + 1], c10 = cm[kBoxW + xl], c11 = cm[kBoxW + xl + 1];
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      int i0, i1;
      float l0;
      gm.xm.at(Xbeg + (i < nx ? i : 0), i0, i1, l0, l1w[i]);
      hm0[i] = fmaf(l1w[i], c01 - c00, c00);
      dm[i] = fmaf(l1w[i], c11 - c10, c10) - hm0[i];
    }
  }
  float s[R][NX], T[R][NX];
#pragma unroll
  for (int j = 0; j < R; ++j)
#pragma unroll
    for (int i = 0; i < NX; ++i) { s[j][i] = 0.f; T[j][i] = 0.f; }

  const int n_chunks = (C + kKC - 1) / kKC;
  for (int k = 0; k < n_chunks; ++k) {
    const int slot = k % kFwdStages;
    const int c_lo = k * kKC;
    const int cc = (C - c_lo) < kKC ? (C - c_lo) : kKC;
    mbar_wait(&bars[slot], (k / kFwdStages) & 1);
    const float* stage = stages + slot * kStageFloats;
    const float* Sp = stage + xl;
#pragma unroll 2
    for (int c = 0; c < cc; ++c) {
      const float v00 = Sp[0] * kLog2e, v01 = Sp[1] * kLog2e;
      const float v10 = Sp[kBoxW] * kLog2e, v11 = Sp[kBoxW + 1] * kLog2e;
      Sp += 2 * kBoxW;
      const float dv0 = v01 - v00, dv1 = v11 - v10;
#pragma unroll
      for (int i = 0; i < NX; ++i) {
        const float h0 = fmaf(l1w[i], dv0, v00);
        const float h1 = fmaf(l1w[i], dv1, v10);
        const float E = h0 - hm0[i];
        const float D = (h1 - h0) - dm[i];
#pragma unroll
        for (int j = 0; j < R; ++j) s[j][i] += ex2_approx(fmaf(l1h[j], D, E));
      }
    }
    // label-class logit (minus M) for the pixels whose label lives in this chunk
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      if (i < nx) {
#pragma unroll
        for (int j = 0; j < R; ++j) {
          const unsigned lc = (unsigned)lab_w[j * kRowBuf + off + i] - (unsigned)c_lo;
          if (lc < (unsigned)cc) {
            const float* q = stage + lc * (2 * kBoxW) + xl;
            const float v00 = q[0] * kLog2e, v01 = q[1] * kLog2e, v10 = q[kBoxW] * kLog2e, v11 = q[kBoxW + 1] * kLog2e;
            const float h0 = fmaf(l1w[i], v01 - v00, v00);
            const float h1 = fmaf(l1w[i], v11 - v10, v10);
            T[j][i] = fmaf(l1h[j], (h1 - h0) - dm[i], h0 - hm0[i]);
          }
        }
      }
    }
    __syncthreads();  // everyone is done with this slot
    if (threadIdx.x == 0 && k + kFwdStages < n_chunks) {
      mbar_expect_tx(&bars[slot], kStageBytes);
      tma_load_4d(stages + slot * kStageFloats, map, &bars[slot], xa, g, (k + kFwdStages) * kKC, b);
    }
  }

  // finalize: loss, lse, statistics; rows leave through the warp's row buffer
#pragma unroll
  for (int j = 0; j < R; ++j) {
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      if (i < nx) {
        const int lab = lab_w[j * kRowBuf + off + i];
        const float lg = lg2_approx(s[j][i]);
        const float M2 = fmaf(l1h[j], dm[i], hm0[i]);
        const bool valid = lab != 255;
        const float l = valid ? (lg - T[j][i]) * kLn2 : 0.f;
        rb[off + i] = l;
        rb[kRowBuf + off + i] = (M2 + lg) * kLn2;
        st.n_valid += valid ? 1u : 0u;
        if (l > thresh) { ++st.n_hard; st.sum_hard += l; }
        ++st.n_px;
      }
    }
    __syncwarp();
    const int64_t rowbase = ((int64_t)b * gm.H + (Ys + j)) * gm.W + Xw0;
    for (int k = lane; k < nw; k += 32) {
      a.loss_px[rowbase + k] = rb[k];
      a.lse_px[rowbase + k] = rb[kRowBuf + k];
    }
    __syncwarp();
  }
}

template <typename L>
__global__ void __launch_bounds__(kT)
up_ce_fwd_tma_kernel(const __grid_constant__ TmaMaps maps, const FwdArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const Geom& gm = a.gm;
  const int b = blockIdx.z, g = blockIdx.y;
  const int xa = blockIdx.x * kT;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  const int Ys = first_dst_ge(gm.ym, g, gm.H);
  const int Ye = first_dst_ge(gm.ym, g + 1, gm.H);
  const int R = Ye - Ys;
  if (R <= 0) return;
  const L* labels = (const L*)a.labels;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  const int x = xa + threadIdx.x;
  const bool active = x <= gm.w - 1;
  const int Xbeg = active ? first_dst_ge(gm.xm, x, gm.W) : gm.W;
  const int Xend = active ? first_dst_ge(gm.xm, x + 1, gm.W) : gm.W;
  const int nx = Xend - Xbeg;
  const int Xw0 = __shfl_sync(0xffffffffu, Xbeg, 0);
  const int Xw1 = __shfl_sync(0xffffffffu, Xend, 31);
  const int nw = Xw1 - Xw0;

  if (d < 0 || d >= a.src.n_datasets) {
    // image outside every dataset: not part of the loss vector (sentinel -1), but
    // its labels still count in n_min (ohem_ce_loss.py:52 uses all labels).
    unsigned n_valid = 0;
    for (int Y = Ys; Y < Ye; ++Y)
      for (int k = lane; k < nw; k += 32) {
        const int64_t p = ((int64_t)b * gm.H + Y) * gm.W + Xw0 + k;
        a.loss_px[p] = -1.0f;
        a.lse_px[p] = 0.f;
        n_valid += (load_label<L>(labels, p) != a.ignore) ? 1u : 0u;
      }
    if (threadIdx.x == 0 && blockIdx.x == 0 && g == 0) atomicOr(a.err_flag, MDSEG_ERR_DATASET_ID);
    block_accumulate_stats(a.states, n_valid, 0u, 0.0, 0u);
    return;
  }
  const int C = a.src.C[d];
  mdseg_ohem_state* st_dev = a.states + (a.src.seg_per_dataset ? d : 0);
  const float thresh = st_dev->thresh;
  const CUtensorMap* map = &maps.m[d];

  // shared memory carve-up (stages first: TMA destinations need 128-byte alignment)
  float* stages = reinterpret_cast<float*>(smem_raw);
  float* cm = stages + kFwdStages * kStageFloats;     // [2][kBoxW]
  float* rowbuf = cm + 2 * kBoxW;                     // [kNW][2][kRowBuf]
  uint8_t* labbuf = reinterpret_cast<uint8_t*>(rowbuf + kNW * 2 * kRowBuf);  // [kNW][kMaxR][kRowBuf]
  uint64_t* bars = reinterpret_cast<uint64_t*>(labbuf + kNW * kMaxR * kRowBuf);

  const int n_chunks = (C + kKC - 1) / kKC;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kFwdStages; ++s) mbar_init(&bars[s], 1);
    mbar_fence_init();
    for (int s = 0; s < kFwdStages && s < n_chunks; ++s) {
      mbar_expect_tx(&bars[s], kStageBytes);
      tma_load_4d(stages + s * kStageFloats, map, &bars[s], xa, g, s * kKC, b);
    }
  }
  // channel maxima of the two rows (zero outside the image, matching the TMA zero fill)
  for (int e = threadIdx.x; e < 2 * kBoxW; e += kT) {
    const int r = e / kBoxW, xl = e - r * kBoxW;
    const int yy = g + r, xx = xa + xl;
    float v = 0.f;
    if (yy <= gm.h - 1 && xx <= gm.w - 1) v = a.src.cmax[((int64_t)b * gm.h + yy) * gm.w + xx] * kLog2e;
    cm[e] = v;
  }
  int err = 0;
  uint8_t* lab_w = labbuf + warp * (kMaxR * kRowBuf);
  stage_labels<L>(lab_w, labels, (int64_t)b * gm.H + Ys, gm.W, R, Xw0, nw, C, a.ignore, err);
  __syncthreads();

  int nxw = nx;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) nxw = max(nxw, __shfl_xor_sync(0xffffffffu, nxw, o));
  // every warp takes the same branch sequence w.r.t. __syncthreads inside fwd_tile: NX is
  // decided per CTA (max over warps) so that the barrier counts match
  __shared__ int s_nx;
  if (threadIdx.x == 0) s_nx = 0;
  __syncthreads();
  if (lane == 0) atomicMax(&s_nx, nxw);
  __syncthreads();
  const int nx_cta = s_nx;

  Stats st;
  float* rb = rowbuf + warp * (2 * kRowBuf);
#define MDSEG_CASE(RR, NN)                                                                                        \
  fwd_tile<L, RR, NN>(a, map, C, b, g, Ys, xa, threadIdx.x, Xbeg, nx, Xw0, nw, stages, bars, cm, lab_w, rb, thresh, st)
  if (nx_cta <= 4) {
    switch (R) {
      case 1: MDSEG_CASE(1, 4); break;
      case 2: MDSEG_CASE(2, 4); break;
      case 3: MDSEG_CASE(3, 4); break;
      case 4: MDSEG_CASE(4, 4); break;
      default: MDSEG_CASE(5, 4); break;
    }
  } else {
    switch (R) {
      case 1: MDSEG_CASE(1, 5); break;
      case 2: MDSEG_CASE(2, 5); break;
      case 3: MDSEG_CASE(3, 5); break;
      case 4: MDSEG_CASE(4, 5); break;
      default: MDSEG_CASE(5, 5); break;
    }
  }
#undef MDSEG_CASE
  if (err) atomicOr(a.err_flag, err);
  block_accumulate_stats(st_dev, st.n_valid, st.n_hard, (double)st.sum_hard, st.n_px);
}

// =================================================================================================
// backward
// =================================================================================================
template <typename L, int R, int NX>
__device__ __forceinline__ void bwd_tile(const BwdArgs& a, const CUtensorMap* map, int C, int b, int g, int Ys,
                                         int box_x0, int xl, int x, int x_end, int Xbeg, int nx, int Xw0, int nw, bool own,
                                         float* stages, uint64_t* bars, float* O, const uint8_t* lab_w, float* rb,
                                         const SelParams& sp, float* dA, float* dB, bool fold_down) {
  const Geom& gm = a.gm;
  const int lane = threadIdx.x & 31;
  const int off = Xbeg - Xw0;
  const int64_t hw = (int64_t)gm.h * gm.w;
  const bool fold_right = (x == gm.w - 1);
  const float wabs = fabsf(sp.w), wsign = sp.w < 0.f ? -1.f : 1.f;
  const float log2w = log2f(wabs);
  float l1w[NX], l1h[R];
#pragma unroll
  for (int j = 0; j < R; ++j) {
    int i0, i1;
    float l0;
    gm.ym.at(Ys + j, i0, i1, l0, l1h[j]);
  }
#pragma unroll
  for (int i = 0; i < NX; ++i) {
    int i0, i1;
    float l0;
    gm.xm.at(Xbeg + (i < nx ? i : 0), i0, i1, l0, l1w[i]);
  }
  // lw2 = lse*log2e - log2(w) for selected valid pixels, +inf otherwise (ex2(-inf) = 0)
  float lw2[R][NX];
#pragma unroll
  for (int j = 0; j < R; ++j) {
    const int64_t rowbase = ((int64_t)b * gm.H + (Ys + j)) * gm.W + Xw0;
    for (int k = lane; k < nw; k += 32) {
      rb[k] = a.loss_px[rowbase + k];
      rb[kRowBuf + k] = a.lse_px[rowbase + k];
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      lw2[j][i] = __int_as_float(0x7f800000);
      if (i < nx) {
        const bool valid = lab_w[j * kRowBuf + off + i] != 255;
        if (valid && wabs > 0.f && is_selected(sp, rb[off + i])) lw2[j][i] = fmaf(rb[kRowBuf + off + i], kLog2e, -log2w);
      }
    }
    __syncwarp();
  }

  const int n_chunks = (C + kKC - 1) / kKC;
  for (int k = 0; k < n_chunks; ++k) {
    const int slot = k % kBwdStages;
    const int c_lo = k * kKC;
    const int cc = (C - c_lo) < kKC ? (C - c_lo) : kKC;
    mbar_wait(&bars[slot], (k / kBwdStages) & 1);
    const float* stage = stages + slot * kStageFloats;
    const float* Sp = stage + xl;
    for (int c = 0; c < cc; ++c) {
      const float v00 = Sp[0] * kLog2e, v01 = Sp[1] * kLog2e;
      const float v10 = Sp[kBoxW] * kLog2e, v11 = Sp[kBoxW + 1] * kLog2e;
      Sp += 2 * kBoxW;
      const float dv0 = v01 - v00, dv1 = v11 - v10;
      float CU = 0.f, ur = 0.f, CL = 0.f, lr = 0.f;
#pragma unroll
      for (int i = 0; i < NX; ++i) {
        const float h0 = fmaf(l1w[i], dv0, v00);
        const float dd = fmaf(l1w[i], dv1, v10) - h0;
        float t0 = 0.f, t1 = 0.f;
#pragma unroll
        for (int j = 0; j < R; ++j) {
          const float e = ex2_approx(fmaf(l1h[j], dd, h0) - lw2[j][i]);
          t0 += e;
          t1 = fmaf(l1h[j], e, t1);
        }
        const float cu = t0 - t1;
        CU += cu; ur = fmaf(l1w[i], cu, ur);
        CL += t1; lr = fmaf(l1w[i], t1, lr);
      }
      float uo = CU - ur, lo = CL - lr;
      if (fold_right) { uo = CU; lo = CL; ur = 0.f; lr = 0.f; }  // x == w-1: x1 == x0
      float gu = __shfl_up_sync(0xffffffffu, ur, 1);
      float gl = __shfl_up_sync(0xffffffffu, lr, 1);
      if (lane == 0) { gu = 0.f; gl = 0.f; }
      if (own) {  // the halo lane shares its column with the previous warp's last own cell
        O[(c * 2 + 0) * kBoxW + xl] = (uo + gu) * wsign;
        O[(c * 2 + 1) * kBoxW + xl] = (lo + gl) * wsign;
      }
    }
    __syncwarp();
    // -w*[c == label]: one scatter per pixel.  phase 0 -> own cell, phase 1 -> right cell
#pragma unroll
    for (int ph = 0; ph < 2; ++ph) {
#pragma unroll
      for (int i = 0; i < NX; ++i) {
        if (i < nx) {
#pragma unroll
          for (int j = 0; j < R; ++j) {
            const unsigned lc = (unsigned)lab_w[j * kRowBuf + off + i] - (unsigned)c_lo;
            if (lc < (unsigned)cc && lw2[j][i] < 3.0e38f) {
              const float wu = sp.w * (1.f - l1h[j]), wl = sp.w * l1h[j];
              if (ph == 0) {
                if (own) {
                  const float fo = fold_right ? 1.f : (1.f - l1w[i]);
                  O[(lc * 2 + 0) * kBoxW + xl] -= wu * fo;
                  O[(lc * 2 + 1) * kBoxW + xl] -= wl * fo;
                }
              } else if (!fold_right && lane < 31) {
                O[(lc * 2 + 0) * kBoxW + xl + 1] -= wu * l1w[i];
                O[(lc * 2 + 1) * kBoxW + xl + 1] -= wl * l1w[i];
              }
            }
          }
        }
      }
      __syncwarp();
    }
    // the warp's own cells leave as plain stores: plane A row g, plane B row g+1
    if (own) {
      for (int c = 0; c < cc; ++c) {
        float u = O[(c * 2 + 0) * kBoxW + xl];
        const float lw = O[(c * 2 + 1) * kBoxW + xl];
        if (fold_down) u += lw;
        dA[(int64_t)(c_lo + c) * hw + (int64_t)g * gm.w + x] = u;
        if (!fold_down) dB[(int64_t)(c_lo + c) * hw + (int64_t)(g + 1) * gm.w + x] = lw;
        if (g == 0) dB[(int64_t)(c_lo + c) * hw + x] = 0.f;  // row 0 of plane B has no producer
      }
    }
    __syncthreads();  // slot and O tile free
    if (threadIdx.x == 0 && k + kBwdStages < n_chunks) {
      mbar_expect_tx(&bars[slot], kStageBytes);
      tma_load_4d(stages + slot * kStageFloats, map, &bars[slot], box_x0, g, (k + kBwdStages) * kKC, b);
    }
  }
  (void)x_end;
}

template <typename L>
__global__ void __launch_bounds__(kT)
up_ce_bwd_tma_kernel(const __grid_constant__ TmaMaps maps, const BwdArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const Geom& gm = a.gm;
  const int b = blockIdx.z, g = blockIdx.y;
  constexpr int kOwn = kNW * kOwnPerWarp;  // owned cells per CTA
  const int xa = blockIdx.x * kOwn;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  if (d < 0 || d >= a.src.n_datasets) return;  // no gradient planes for this image
  const int C = a.src.C[d];
  float* dA = (float*)a.dstA.base[d] + (int64_t)b * a.dstA.image_stride[d];
  float* dB = (float*)a.dstB.base[d] + (int64_t)b * a.dstB.image_stride[d];
  mdseg_ohem_state* st = a.states + (a.src.seg_per_dataset ? d : 0);
  const L* labels = (const L*)a.labels;
  const CUtensorMap* map = &maps.m[d];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t hw = (int64_t)gm.h * gm.w;

  SelParams sp;
  sp.thresh = st->thresh; sp.kth = st->kth; sp.mode = st->mode;
  sp.w = (a.grad_out ? a.grad_out[a.src.seg_per_dataset ? d : 0] : 1.f) * a.grad_scale * st->inv_n_sel;

  const int Ys = first_dst_ge(gm.ym, g, gm.H);
  const int Ye = first_dst_ge(gm.ym, g + 1, gm.H);
  const int R = Ye - Ys;
  const bool fold_down = (g == gm.h - 1);  // last low-res row: y1 == y0

  // warps overlap by one cell: lane 0 is the left halo of the warp's 31 own cells
  const int x = xa + warp * kOwnPerWarp + lane - 1;
  // staged column of this cell.  The TMA box must start at or left of the halo cell xa-1, and its
  // innermost start coordinate has to be a multiple of 16 bytes: an unaligned (or negative) start
  // raises "illegal instruction" on B200 (fp32, SWIZZLE_NONE, driver 580, CUDA 12.9).  xa is a multiple
  // of 124, so the box starts 4 cells left of xa (at 0 for the first CTA of a row).
  static_assert((kNW * kOwnPerWarp) % 4 == 0, "box start must stay 16-byte aligned");
  const int box_x0 = xa > 0 ? xa - 4 : 0;
  const int xl = (x - box_x0) > 0 ? (x - box_x0) : 0;
  const int x_end = (xa + kOwn < gm.w) ? xa + kOwn : gm.w;
  const bool in_img = (x >= 0) && (x <= gm.w - 1) && (x < x_end);
  const bool own = in_img && lane >= 1;
  const int Xbeg = in_img ? first_dst_ge(gm.xm, x, gm.W) : -1;
  const int Xend = in_img ? first_dst_ge(gm.xm, x + 1, gm.W) : -1;
  const int nx = in_img ? Xend - Xbeg : 0;
  // the warp's label-column span: first in-image lane .. last in-image lane
  const unsigned in_mask = __ballot_sync(0xffffffffu, in_img);
  int Xw0 = 0, nw = 0;
  if (in_mask) {
    Xw0 = __shfl_sync(0xffffffffu, Xbeg, __ffs(in_mask) - 1);
    nw = __shfl_sync(0xffffffffu, Xend, 31 - __clz(in_mask)) - Xw0;
  }

  if (R <= 0) {  // no label row interpolates from (g, g+1): zero planes
    if (own)
      for (int c = 0; c < C; ++c) {
        dA[(int64_t)c * hw + (int64_t)g * gm.w + x] = 0.f;
        if (!fold_down) dB[(int64_t)c * hw + (int64_t)(g + 1) * gm.w + x] = 0.f;
        if (g == 0) dB[(int64_t)c * hw + x] = 0.f;
      }
    return;
  }

  float* stages = reinterpret_cast<float*>(smem_raw);
  float* O = stages + kBwdStages * kStageFloats;      // [kKC][2][kBoxW]
  float* rowbuf = O + kStageFloats;                   // [kNW][2][kRowBuf]
  uint8_t* labbuf = reinterpret_cast<uint8_t*>(rowbuf + kNW * 2 * kRowBuf);
  uint64_t* bars = reinterpret_cast<uint64_t*>(labbuf + kNW * kMaxR * kRowBuf);

  const int n_chunks = (C + kKC - 1) / kKC;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kBwdStages; ++s) mbar_init(&bars[s], 1);
    mbar_fence_init();
    for (int s = 0; s < kBwdStages && s < n_chunks; ++s) {
      mbar_expect_tx(&bars[s], kStageBytes);
      tma_load_4d(stages + s * kStageFloats, map, &bars[s], box_x0, g, s * kKC, b);
    }
  }
  int err = 0;
  uint8_t* lab_w = labbuf + warp * (kMaxR * kRowBuf);
  stage_labels<L>(lab_w, labels, (int64_t)b * gm.H + Ys, gm.W, R, Xw0, nw, C, a.ignore, err);

  int nxw = nx;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) nxw = max(nxw, __shfl_xor_sync(0xffffffffu, nxw, o));
  __shared__ int s_nx;
  if (threadIdx.x == 0) s_nx = 0;
  __syncthreads();
  if (lane == 0) atomicMax(&s_nx, nxw);
  __syncthreads();
  const int nx_cta = s_nx;

  float* rb = rowbuf + warp * (2 * kRowBuf);
#define MDSEG_CASE(RR, NN)                                                                                         \
  bwd_tile<L, RR, NN>(a, map, C, b, g, Ys, box_x0, xl, x, x_end, Xbeg, nx, Xw0, nw, own, stages, bars, O, lab_w, rb, sp, \
                      dA, dB, fold_down)
  if (nx_cta <= 4) {
    switch (R) {
      case 1: MDSEG_CASE(1, 4); break;
      case 2: MDSEG_CASE(2, 4); break;
      case 3: MDSEG_CASE(3, 4); break;
      case 4: MDSEG_CASE(4, 4); break;
      default: MDSEG_CASE(5, 4); break;
    }
  } else {
    switch (R) {
      case 1: MDSEG_CASE(1, 5); break;
      case 2: MDSEG_CASE(2, 5); break;
      case 3: MDSEG_CASE(3, 5); break;
      case 4: MDSEG_CASE(4, 5); break;
      default: MDSEG_CASE(5, 5); break;
    }
  }
#undef MDSEG_CASE
}

// =================================================================================================
// host side
// =================================================================================================
bool tma_applicable(const mdseg_src_table& src, const Geom& gm) {
  if (src.dtype != MDSEG_F32 || src.cmax == nullptr) return false;
  if (gm.w % 4 != 0 || gm.h < 1) return false;
  if (gm.ym.scale < 0.2002f || gm.xm.scale < 0.2002f) return false;  // at most 5 label rows / columns per cell
  for (int i = 0; i < src.n_datasets; ++i) {
    if (src.C[i] > 254) return false;  // labels are staged as bytes
    if (((uintptr_t)src.base[i] & 15) != 0 || (src.image_stride[i] % 4) != 0) return false;
  }
  return tma::encode_fn() != nullptr;
}

int make_maps(const mdseg_src_table& src, const Geom& gm, int n_images, TmaMaps* out) {
  tma::EncodeTiledFn enc = tma::encode_fn();
  if (int rc = tma::bind_primary_context()) return rc;
  for (int i = 0; i < src.n_datasets; ++i) {
    const int calloc = src.C_alloc[i] > 0 ? src.C_alloc[i] : src.C[i];
    cuuint64_t dims[4] = {(cuuint64_t)gm.w, (cuuint64_t)gm.h, (cuuint64_t)calloc, (cuuint64_t)n_images};
    cuuint64_t strides[3] = {(cuuint64_t)gm.w * 4, (cuuint64_t)gm.h * gm.w * 4, (cuuint64_t)src.image_stride[i] * 4};
    cuuint32_t box[4] = {(cuuint32_t)kBoxW, 2, (cuuint32_t)kKC, 1};
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

constexpr size_t kFwdSmem = (size_t)kFwdStages * kStageBytes + 2 * kBoxW * 4 + kNW * 2 * kRowBuf * 4 +
                            kNW * kMaxR * kRowBuf + kFwdStages * 8 + 64;
constexpr size_t kBwdSmem = (size_t)(kBwdStages + 1) * kStageBytes + kNW * 2 * kRowBuf * 4 + kNW * kMaxR * kRowBuf +
                            kBwdStages * 8 + 64;

template <typename L>
int launch_fwd(const TmaMaps& maps, const FwdArgs& a, int n_images, cudaStream_t s) {
  auto k = up_ce_fwd_tma_kernel<L>;
  MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFwdSmem));
  dim3 grid((unsigned)((a.gm.w + kT - 1) / kT), (unsigned)a.gm.h, (unsigned)n_images);
  k<<<grid, kT, kFwdSmem, s>>>(maps, a);
  MDSEG_LAUNCH_OK();
  return 0;
}
template <typename L>
int launch_bwd(const TmaMaps& maps, const BwdArgs& a, int n_images, cudaStream_t s) {
  auto k = up_ce_bwd_tma_kernel<L>;
  MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdSmem));
  constexpr int kOwn = kNW * kOwnPerWarp;
  dim3 grid((unsigned)((a.gm.w + kOwn - 1) / kOwn), (unsigned)a.gm.h, (unsigned)n_images);
  k<<<grid, kT, kBwdSmem, s>>>(maps, a);
  MDSEG_LAUNCH_OK();
  return 0;
}

}  // namespace

int up_ce_fwd_tma(const FwdArgs& a, int label_dtype, int n_images, cudaStream_t s) {
  if (!tma_applicable(a.src, a.gm)) return -1;
  TmaMaps maps;
  if (int rc = make_maps(a.src, a.gm, n_images, &maps)) return rc;
  if (!a.src.cmax_ready)
    if (int rc = tma::channel_max(a.src, a.dataset_ids, n_images, (int64_t)a.gm.h * a.gm.w, s)) return rc;
  switch (label_dtype) {
    case MDSEG_U8: return launch_fwd<uint8_t>(maps, a, n_images, s);
    case MDSEG_I32: return launch_fwd<int32_t>(maps, a, n_images, s);
    case MDSEG_I64: return launch_fwd<int64_t>(maps, a, n_images, s);
  }
  return -1;
}

int up_ce_bwd_tma(const BwdArgs& a, int label_dtype, int n_images, cudaStream_t s) {
  if (!tma_applicable(a.src, a.gm)) return -1;
  TmaMaps maps;
  if (int rc = make_maps(a.src, a.gm, n_images, &maps)) return rc;
  switch (label_dtype) {
    case MDSEG_U8: return launch_bwd<uint8_t>(maps, a, n_images, s);
    case MDSEG_I32: return launch_bwd<int32_t>(maps, a, n_images, s);
    case MDSEG_I64: return launch_bwd<int64_t>(maps, a, n_images, s);
  }
  return -1;
}

}  // namespace mdseg
