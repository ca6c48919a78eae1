// up_ce.cu — fused bilinear upsample (align_corners=True) + per-pixel
// cross-entropy, forward and adjoint (SURVEY §8 rows a6, a7, a9, a10).
//
// Reference work replaced (lib/loss/loss_cross_datasets.py:1007,1051 and
// lib/loss/ohem_ce_loss.py:27,61, plus their autograd replay):
//   up   = F.interpolate(remap_logit, size=(H,W), mode="bilinear", align_corners=True)
//   loss = CrossEntropyLoss(ignore_index=255, reduction='none')(up, labels)
// ATen materialises the [B,C,H,W] upsampled tensor (2.5 GB for ADE at
// 1024x2048), a second one for log_softmax and a third in the backward, and
// scatters the upsample gradient with atomics.  Here nothing of size C*H*W ever
// exists:
//
//  * CTA = one image, one low-res row g ("row group": all label rows Y whose
//    upper interpolation row is g — 4 or 5 rows at stride 4), 128 low-res cells.
//  * thread = one low-res cell: its 4 corner logits are read once per class from
//    the staged shared-memory tile and reused by the ~4x4 label pixels inside
//    the cell (registers: per-pixel running sums).
//  * softmax shift: the bilinear interpolation M of the per-corner channel maxima
//    is an upper bound of max_c z_c at every pixel (interpolation weights are
//    non-negative and every fp op involved is monotone), so Σ exp(z_c - M) never
//    overflows and needs no online rescaling: one FADD + one MUFU.EX2 + one FADD
//    per (pixel, class).  Tiles are staged pre-multiplied by log2(e).
//  * backward = adjoint in gather form: per class the cell-thread accumulates
//    Σ w·p over its pixels for its own cell and its right neighbour (one
//    shuffle), in two planes (upper row g / lower row g+1); plane A[g] and
//    B[g+1] are written with plain stores — no global atomics, deterministic.
//    The -w·[c==label] term is scattered once per pixel, not once per class.
//
// The per-(pixel,class) cost is ~6 issue slots forward and ~9 backward; HBM
// traffic per label pixel is C*4/16 (low-res logits) + L (label) + 8 (loss, lse).
#include <float.h>
#include <type_traits>

#include "up_ce_internal.cuh"

namespace mdseg {
namespace {

constexpr int kCT = 128;  // threads per CTA = low-res cells per CTA (incl. 1 halo in the backward)
constexpr int kRB = 5;    // label rows per register tile
constexpr int kNB = 5;    // label columns per register tile
constexpr int kWarps = kCT / 32;
constexpr int kRowBuf = 32 * kNB;  // per-warp staging row for coalesced stores

// Stage classes [c_lo, c_lo+cc) of the two low-res rows (g, y1) and columns
// [xlo, xlo+fw) (clamped to w-1) into S2[(c*2+r)*fwp + xl], scaled by log2(e).
template <typename T>
__device__ __forceinline__ void stage_chunk(float* __restrict__ S2, const T* __restrict__ img, int c_lo, int cc, int g,
                                            int y1, int xlo, int fw, int fwp, int h, int w) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t hw = (int64_t)h * w;
  for (int cr = warp; cr < cc * 2; cr += kWarps) {
    const int c = cr >> 1, r = cr & 1;
    const T* row = img + (int64_t)(c_lo + c) * hw + (int64_t)(r ? y1 : g) * w;
    float* dst = S2 + (int64_t)cr * fwp;
    for (int xl = lane; xl < fw; xl += 32) {
      int xg = xlo + xl;
      xg = xg > w - 1 ? w - 1 : xg;
      dst[xl] = to_f32<T>(row[xg]) * kLog2e;
    }
  }
}

// cm[r*fwp + xl] = max_c (log2e * src[c][row r][xlo+xl]) over ALL classes
template <typename T>
__device__ __forceinline__ void channel_max_global(float* __restrict__ cm, const T* __restrict__ img, int C, int g,
                                                   int y1, int xlo, int fw, int fwp, int h, int w) {
  const int64_t hw = (int64_t)h * w;
  for (int e = threadIdx.x; e < 2 * fw; e += kCT) {
    const int r = e / fw, xl = e - r * fw;
    int xg = xlo + xl;
    xg = xg > w - 1 ? w - 1 : xg;
    const T* p = img + (int64_t)(r ? y1 : g) * w + xg;
    float m = -FLT_MAX;
    for (int c = 0; c < C; ++c) m = fmaxf(m, to_f32<T>(p[(int64_t)c * hw]));
    cm[r * fwp + xl] = m * kLog2e;
  }
}
__device__ __forceinline__ void channel_max_smem(float* __restrict__ cm, const float* __restrict__ S2, int C, int fw,
                                                 int fwp) {
  for (int e = threadIdx.x; e < 2 * fw; e += kCT) {
    const int r = e / fw, xl = e - r * fw;
    float m = -FLT_MAX;
    for (int c = 0; c < C; ++c) m = fmaxf(m, S2[(int64_t)(c * 2 + r) * fwp + xl]);
    cm[r * fwp + xl] = m;
  }
}

// ---------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------
template <typename T, typename L, int R>
__device__ __forceinline__ void fwd_rows(const FwdArgs& a, const T* __restrict__ img, int C, int b, int g, int y1,
                                         int Yb, int xlo, int fw, int x, int xl, int Xbeg, int nx, int nx_max,
                                         bool single_chunk, float* S2, float* cm, float* rowbuf, unsigned& n_valid,
                                         unsigned& n_hard, double& sum_hard, unsigned& n_px, int& err, float thresh) {
  const Geom& gm = a.gm;
  const L* labels = (const L*)a.labels;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int fwp = a.fwp;
  float l0h[R], l1h[R];
#pragma unroll
  for (int j = 0; j < R; ++j) {
    int i0, i1;
    gm.ym.at(Yb + j, i0, i1, l0h[j], l1h[j]);
  }
  // first label column of this warp (for the coalesced store of loss / lse)
  const int Xw0 = __shfl_sync(0xffffffffu, Xbeg, 0);

  for (int Xo = 0; Xo < nx_max; Xo += kNB) {
    int nxb = nx - Xo;
    nxb = nxb < 0 ? 0 : (nxb > kNB ? kNB : nxb);
    float l0w[kNB], l1w[kNB];
#pragma unroll
    for (int i = 0; i < kNB; ++i) {
      int i0, i1;
      gm.xm.at(Xbeg + Xo + (i < nxb ? i : 0), i0, i1, l0w[i], l1w[i]);
    }
    float M[R][kNB], s[R][kNB], zl[R][kNB];
    {
      const float c00 = cm[xl], c01 = cm[xl + 1], c10 = cm[fwp + xl], c11 = cm[fwp + xl + 1];
#pragma unroll
      for (int i = 0; i < kNB; ++i) {
        const float h0 = l0w[i] * c00 + l1w[i] * c01;
        const float h1 = l0w[i] * c10 + l1w[i] * c11;
#pragma unroll
        for (int j = 0; j < R; ++j) {
          M[j][i] = l0h[j] * h0 + l1h[j] * h1;
          s[j][i] = 0.f;
          zl[j][i] = 0.f;
        }
      }
    }
    for (int c_lo = 0; c_lo < C; c_lo += a.cc_max) {
      const int cc = (C - c_lo) < a.cc_max ? (C - c_lo) : a.cc_max;
      if (!single_chunk) {
        __syncthreads();
        stage_chunk<T>(S2, img, c_lo, cc, g, y1, xlo, fw, fwp, gm.h, gm.w);
        __syncthreads();
      }
      const float* Sp = S2 + xl;
#pragma unroll 2
      for (int c = 0; c < cc; ++c) {
        const float v00 = Sp[0], v01 = Sp[1], v10 = Sp[fwp], v11 = Sp[fwp + 1];
        Sp += 2 * fwp;
#pragma unroll
        for (int i = 0; i < kNB; ++i) {
          if (i < nxb) {
            const float h0 = l0w[i] * v00 + l1w[i] * v01;
            const float h1 = l0w[i] * v10 + l1w[i] * v11;
#pragma unroll
            for (int j = 0; j < R; ++j) {
              const float z = l0h[j] * h0 + l1h[j] * h1;
              s[j][i] += ex2_approx(z - M[j][i]);
            }
          }
        }
      }
      // logit of the label class, for pixels whose label lives in this chunk
#pragma unroll
      for (int i = 0; i < kNB; ++i) {
        if (i < nxb) {
#pragma unroll
          for (int j = 0; j < R; ++j) {
            const int lab = load_label<L>(labels, ((int64_t)b * gm.H + (Yb + j)) * gm.W + Xbeg + Xo + i);
            const unsigned lc = (unsigned)(lab - c_lo);
            if (lab != a.ignore && lc < (unsigned)cc) {
              const float* q = S2 + (int64_t)lc * 2 * fwp + xl;
              const float h0 = l0w[i] * q[0] + l1w[i] * q[1];
              const float h1 = l0w[i] * q[fwp] + l1w[i] * q[fwp + 1];
              zl[j][i] = l0h[j] * h0 + l1h[j] * h1;
            }
          }
        }
      }
    }
    // finalize: loss / lse, statistics, coalesced stores through the warp row buffer
#pragma unroll
    for (int j = 0; j < R; ++j) {
      float lo[kNB], ls[kNB];
#pragma unroll
      for (int i = 0; i < kNB; ++i) {
        lo[i] = 0.f;
        ls[i] = 0.f;
        if (i < nxb) {
          const int lab = load_label<L>(labels, ((int64_t)b * gm.H + (Yb + j)) * gm.W + Xbeg + Xo + i);
          const float lse2 = M[j][i] + log2f(s[j][i]);
          const bool ign = lab == a.ignore;
          const bool ok = (unsigned)lab < (unsigned)C;
          if (!ign && !ok) err |= MDSEG_ERR_LABEL_RANGE;
          const float l = (ok && !ign) ? (lse2 - zl[j][i]) * kLn2 : 0.f;
          lo[i] = l;
          ls[i] = lse2 * kLn2;
          n_valid += (ok && !ign) ? 1u : 0u;
          if (l > thresh) { ++n_hard; sum_hard += (double)l; }
          ++n_px;
        }
      }
      // The label columns of a warp are contiguous: [Xw0, Xw0 + n_w).  Column
      // tile Xo of every cell is staged, then written row-contiguously.
      const int64_t rowbase = ((int64_t)b * gm.H + (Yb + j)) * gm.W;
      float* rb = rowbuf + warp * (2 * kRowBuf);
      // positions inside the warp's span: cells are laid out back to back
      // only when Xo == 0 and nx <= kNB; in general use direct stores.
      if (nx_max <= kNB) {
        const int off = Xbeg - Xw0;  // < 32*kNB
#pragma unroll
        for (int i = 0; i < kNB; ++i)
          if (i < nxb) { rb[off + i] = lo[i]; rb[kRowBuf + off + i] = ls[i]; }
        __syncwarp();
        const int Xw1 = __shfl_sync(0xffffffffu, Xbeg + nx, 31);
        const int nw = Xw1 - Xw0;
        for (int k = lane; k < nw; k += 32) {
          a.loss_px[rowbase + Xw0 + k] = rb[k];
          a.lse_px[rowbase + Xw0 + k] = rb[kRowBuf + k];
        }
        __syncwarp();
      } else {
#pragma unroll
        for (int i = 0; i < kNB; ++i)
          if (i < nxb) {
            a.loss_px[rowbase + Xbeg + Xo + i] = lo[i];
            a.lse_px[rowbase + Xbeg + Xo + i] = ls[i];
          }
      }
    }
  }
}

template <typename T, typename L>
__global__ void __launch_bounds__(kCT)
up_ce_fwd_kernel(const FwdArgs a) {
  extern __shared__ float smem[];
  const Geom& gm = a.gm;
  const int b = blockIdx.z, g = blockIdx.y;
  const int xa = blockIdx.x * kCT;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  const int Ys = first_dst_ge(gm.ym, g, gm.H);
  const int Ye = first_dst_ge(gm.ym, g + 1, gm.H);
  if (Ys >= Ye) return;
  const L* labels = (const L*)a.labels;

  const int x = xa + threadIdx.x;
  const bool active = x <= gm.w - 1;
  const int Xbeg = active ? first_dst_ge(gm.xm, x, gm.W) : gm.W;
  const int Xend = active ? first_dst_ge(gm.xm, x + 1, gm.W) : gm.W;
  const int nx = Xend - Xbeg;

  unsigned n_valid = 0, n_hard = 0, n_px = 0;
  double sum_hard = 0.0;
  int err = 0;

  if (d < 0 || d >= a.src.n_datasets) {
    // image outside every dataset: not part of the loss vector (sentinel -1), but
    // its labels still count in n_min (ohem_ce_loss.py:52 uses all labels).
    for (int Y = Ys; Y < Ye; ++Y)
      for (int X = Xbeg; X < Xend; ++X) {
        const int64_t p = ((int64_t)b * gm.H + Y) * gm.W + X;
        a.loss_px[p] = -1.0f;
        a.lse_px[p] = 0.f;
        n_valid += (load_label<L>(labels, p) != a.ignore) ? 1u : 0u;
      }
    if (threadIdx.x == 0 && blockIdx.x == 0 && g == 0) atomicOr(a.err_flag, MDSEG_ERR_DATASET_ID);
    block_accumulate_stats(a.states, n_valid, 0u, 0.0, 0u);
    return;
  }
  const int C = a.src.C[d];
  const T* img = (const T*)a.src.base[d] + (int64_t)b * a.src.image_stride[d];
  mdseg_ohem_state* st = a.states + (a.src.seg_per_dataset ? d : 0);
  const float thresh = st->thresh;

  const int y1 = g + ((g < gm.h - 1) ? 1 : 0);
  const int xlo = xa;
  int fw = gm.w - xa;  // cells in this CTA (+1 right neighbour column)
  fw = (fw > kCT ? kCT : fw) + 1;
  const int fwp = a.fwp;
  float* cm = smem;                      // [2][fwp]
  float* rowbuf = cm + 2 * fwp;          // [kWarps][2][kRowBuf]
  float* S2 = rowbuf + kWarps * 2 * kRowBuf;  // [cc_max][2][fwp]
  const bool single_chunk = C <= a.cc_max;
  if (single_chunk) {
    stage_chunk<T>(S2, img, 0, C, g, y1, xlo, fw, fwp, gm.h, gm.w);
    __syncthreads();
    channel_max_smem(cm, S2, C, fw, fwp);
  } else {
    channel_max_global<T>(cm, img, C, g, y1, xlo, fw, fwp, gm.h, gm.w);
  }
  __syncthreads();

  int nx_max = nx;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) nx_max = max(nx_max, __shfl_xor_sync(0xffffffffu, nx_max, o));
  __shared__ int s_nxmax;
  if (threadIdx.x == 0) s_nxmax = 0;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) atomicMax(&s_nxmax, nx_max);
  __syncthreads();
  nx_max = s_nxmax;

  const int xl = threadIdx.x;
  for (int Yb = Ys; Yb < Ye; Yb += kRB) {
    const int R = (Ye - Yb) < kRB ? (Ye - Yb) : kRB;
#define MDSEG_FWD_CASE(RR)                                                                                        \
  case RR:                                                                                                        \
    fwd_rows<T, L, RR>(a, img, C, b, g, y1, Yb, xlo, fw, x, xl, Xbeg, nx, nx_max, single_chunk, S2, cm, rowbuf,   \
                       n_valid, n_hard, sum_hard, n_px, err, thresh);                                             \
    break;
    switch (R) {
      MDSEG_FWD_CASE(1) MDSEG_FWD_CASE(2) MDSEG_FWD_CASE(3) MDSEG_FWD_CASE(4) MDSEG_FWD_CASE(5)
    }
#undef MDSEG_FWD_CASE
  }
  if (err) atomicOr(a.err_flag, err);
  block_accumulate_stats(st, n_valid, n_hard, sum_hard, n_px);
}

// ---------------------------------------------------------------------------
// backward (adjoint)
// ---------------------------------------------------------------------------
// One register tile (R rows x <=kNB columns of the thread's cell) against the
// staged chunk; accumulates into the shared output tile O[(c*2+plane)*fwp + t].
template <typename T, typename L, int R>
__device__ __forceinline__ void bwd_rows(const BwdArgs& a, int C, int c_lo, int cc, int b, int Yb, int Xbeg, int Xo,
                                         int nxb, bool own, bool fold_right, const float* S2, float* O, float* edge,
                                         const SelParams& sp) {
  const Geom& gm = a.gm;
  const L* labels = (const L*)a.labels;
  const int fwp = a.fwp;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  float l0h[R], l1h[R], l0w[kNB], l1w[kNB];
#pragma unroll
  for (int j = 0; j < R; ++j) {
    int i0, i1;
    gm.ym.at(Yb + j, i0, i1, l0h[j], l1h[j]);
  }
#pragma unroll
  for (int i = 0; i < kNB; ++i) {
    int i0, i1;
    gm.xm.at(Xbeg + Xo + (i < nxb ? i : 0), i0, i1, l0w[i], l1w[i]);
  }
  float wgt[R][kNB], lse2[R][kNB];
#pragma unroll
  for (int j = 0; j < R; ++j)
#pragma unroll
    for (int i = 0; i < kNB; ++i) {
      wgt[j][i] = 0.f;
      lse2[j][i] = 0.f;
      if (i < nxb) {
        const int64_t p = ((int64_t)b * gm.H + (Yb + j)) * gm.W + Xbeg + Xo + i;
        const int lab = load_label<L>(labels, p);
        const bool valid = (lab != a.ignore) && ((unsigned)lab < (unsigned)C);
        const bool sel = is_selected(sp, a.loss_px[p]);
        wgt[j][i] = (sel && valid) ? sp.w : 0.f;
        lse2[j][i] = a.lse_px[p] * kLog2e;
      }
    }

  const float* Sp = S2 + t;
  for (int c = 0; c < cc; ++c) {
    const float v00 = Sp[0], v01 = Sp[1], v10 = Sp[fwp], v11 = Sp[fwp + 1];
    Sp += 2 * fwp;
    float uo = 0.f, ur = 0.f, lo = 0.f, lr = 0.f;  // upper/lower plane, own/right cell
#pragma unroll
    for (int i = 0; i < kNB; ++i) {
      if (i < nxb) {
        const float h0 = l0w[i] * v00 + l1w[i] * v01;
        const float h1 = l0w[i] * v10 + l1w[i] * v11;
        float cu = 0.f, cl = 0.f;
#pragma unroll
        for (int j = 0; j < R; ++j) {
          const float z = l0h[j] * h0 + l1h[j] * h1;
          const float e = wgt[j][i] * ex2_approx(z - lse2[j][i]);
          cu = fmaf(l0h[j], e, cu);
          cl = fmaf(l1h[j], e, cl);
        }
        uo = fmaf(l0w[i], cu, uo); ur = fmaf(l1w[i], cu, ur);
        lo = fmaf(l0w[i], cl, lo); lr = fmaf(l1w[i], cl, lr);
      }
    }
    if (fold_right) { uo += ur; lo += lr; ur = 0.f; lr = 0.f; }  // x == w-1: x1 == x0
    // right-cell parts travel one lane up; the warp edge goes through smem
    float gu = __shfl_up_sync(0xffffffffu, ur, 1);
    float gl = __shfl_up_sync(0xffffffffu, lr, 1);
    if (lane == 0) { gu = 0.f; gl = 0.f; }
    if (lane == 31) { edge[(c * 2 + 0) * kWarps + warp] = ur; edge[(c * 2 + 1) * kWarps + warp] = lr; }
    if (own) {
      O[(int64_t)(c * 2 + 0) * fwp + t] += uo + gu;
      O[(int64_t)(c * 2 + 1) * fwp + t] += lo + gl;
    }
  }
}

template <typename T, typename L>
__global__ void __launch_bounds__(kCT)
up_ce_bwd_kernel(const BwdArgs a) {
  extern __shared__ float smem[];
  const Geom& gm = a.gm;
  const int b = blockIdx.z, g = blockIdx.y;
  const int n_own = kCT - 1;               // thread 0 is the left halo cell
  const int xa = blockIdx.x * n_own;       // first owned cell
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  if (d < 0 || d >= a.src.n_datasets) return;  // no gradient planes for this image
  const int C = a.src.C[d];
  const T* img = (const T*)a.src.base[d] + (int64_t)b * a.src.image_stride[d];
  float* dA = (float*)a.dstA.base[d] + (int64_t)b * a.dstA.image_stride[d];
  float* dB = (float*)a.dstB.base[d] + (int64_t)b * a.dstB.image_stride[d];
  mdseg_ohem_state* st = a.states + (a.src.seg_per_dataset ? d : 0);
  const L* labels = (const L*)a.labels;

  SelParams sp;
  sp.thresh = st->thresh; sp.kth = st->kth; sp.mode = st->mode;
  sp.w = (a.grad_out ? a.grad_out[a.src.seg_per_dataset ? d : 0] : 1.f) * a.grad_scale * st->inv_n_sel;

  const int Ys = first_dst_ge(gm.ym, g, gm.H);
  const int Ye = first_dst_ge(gm.ym, g + 1, gm.H);
  const int y1 = g + ((g < gm.h - 1) ? 1 : 0);
  const bool fold_down = (y1 == g);  // last low-res row: lower plane folds into the upper one

  const int t = threadIdx.x;
  const int x = xa - 1 + t;  // this thread's cell
  const int x_end = (xa + n_own < gm.w) ? xa + n_own : gm.w;  // owned cells: [xa, x_end)
  const bool in_img = (x >= 0) && (x <= gm.w - 1) && (x < x_end);
  const bool own = in_img && (t >= 1);
  const bool fold_right = in_img && (x == gm.w - 1);
  const int Xbeg = in_img ? first_dst_ge(gm.xm, x, gm.W) : gm.W;
  const int Xend = in_img ? first_dst_ge(gm.xm, x + 1, gm.W) : gm.W;
  const int nx = Xend - Xbeg;

  __shared__ int s_nxmax;
  if (t == 0) s_nxmax = 0;
  __syncthreads();
  if (nx > 0) atomicMax(&s_nxmax, nx);
  __syncthreads();
  const int nx_max = s_nxmax;

  const int xlo = xa - 1;                   // staged column of thread t is xlo + t (clamped to [0, w-1])
  const int fw = kCT + 1;
  const int fwp = a.fwp;
  float* edge = smem;                                   // [cc_max][2][kWarps]
  float* O = edge + a.cc_max * 2 * kWarps;              // [cc_max][2][fwp]
  float* S2 = O + (int64_t)a.cc_max * 2 * fwp;          // [cc_max][2][fwp]
  const int64_t hw = (int64_t)gm.h * gm.w;

  bool first_tile = true;
  const int n_rows = Ye - Ys;
  // at least one pass so that empty groups still write zero planes
  const int n_rb = n_rows > 0 ? (n_rows + kRB - 1) / kRB : 1;
  const int n_cb = nx_max > 0 ? (nx_max + kNB - 1) / kNB : 1;
  for (int rbi = 0; rbi < n_rb; ++rbi) {
    const int Yb = Ys + rbi * kRB;
    int R = Ye - Yb;
    R = R < 0 ? 0 : (R > kRB ? kRB : R);
    for (int cbi = 0; cbi < n_cb; ++cbi) {
      const int Xo = cbi * kNB;
      int nxb = nx - Xo;
      nxb = nxb < 0 ? 0 : (nxb > kNB ? kNB : nxb);
      for (int c_lo = 0; c_lo < C; c_lo += a.cc_max) {
        const int cc = (C - c_lo) < a.cc_max ? (C - c_lo) : a.cc_max;
        __syncthreads();
        // stage with the left halo: column index t <-> cell xlo + t, clamped on both sides
        {
          const int lane = t & 31, warp = t >> 5;
          for (int cr = warp; cr < cc * 2; cr += kWarps) {
            const int c = cr >> 1, r = cr & 1;
            const T* row = img + (int64_t)(c_lo + c) * hw + (int64_t)(r ? y1 : g) * gm.w;
            float* dst = S2 + (int64_t)cr * fwp;
            for (int xl = lane; xl < fw; xl += 32) {
              int xg = xlo + xl;
              xg = xg < 0 ? 0 : (xg > gm.w - 1 ? gm.w - 1 : xg);
              dst[xl] = to_f32<T>(row[xg]) * kLog2e;
            }
          }
          for (int e = t; e < cc * 2 * fwp; e += kCT) O[e] = 0.f;
          for (int e = t; e < cc * 2 * kWarps; e += kCT) edge[e] = 0.f;
        }
        __syncthreads();
        if (R > 0) {
#define MDSEG_BWD_CASE(RR)                                                                                     \
  case RR:                                                                                                     \
    bwd_rows<T, L, RR>(a, C, c_lo, cc, b, Yb, Xbeg, Xo, nxb, own, fold_right, S2, O, edge, sp);      \
    break;
          switch (R) { MDSEG_BWD_CASE(1) MDSEG_BWD_CASE(2) MDSEG_BWD_CASE(3) MDSEG_BWD_CASE(4) MDSEG_BWD_CASE(5) }
#undef MDSEG_BWD_CASE
        }
        __syncthreads();
        // warp-edge contributions: lane 0 of warp k (k >= 1) receives from lane 31 of warp k-1
        if ((t & 31) == 0 && t > 0 && own) {
          const int wprev = (t >> 5) - 1;
          for (int c = 0; c < cc; ++c) {
            O[(int64_t)(c * 2 + 0) * fwp + t] += edge[(c * 2 + 0) * kWarps + wprev];
            O[(int64_t)(c * 2 + 1) * fwp + t] += edge[(c * 2 + 1) * kWarps + wprev];
          }
        }
        __syncthreads();
        // -w*[c == label] term, one scatter per pixel: phase 0 own cell, phase 1 right cell
        for (int ph = 0; ph < 2; ++ph) {
          if (R > 0 && nxb > 0) {
            for (int j = 0; j < R; ++j) {
              int i0, i1;
              float lh0, lh1;
              gm.ym.at(Yb + j, i0, i1, lh0, lh1);
              for (int i = 0; i < nxb; ++i) {
                const int64_t p = ((int64_t)b * gm.H + (Yb + j)) * gm.W + Xbeg + Xo + i;
                const int lab = load_label<L>(labels, p);
                const unsigned lc = (unsigned)(lab - c_lo);
                if (lab == a.ignore || (unsigned)lab >= (unsigned)C || lc >= (unsigned)cc) continue;
                if (!is_selected(sp, a.loss_px[p])) continue;
                float lw0, lw1;
                int j0, j1;
                gm.xm.at(Xbeg + Xo + i, j0, j1, lw0, lw1);
                const float wu = sp.w * lh0, wl = sp.w * lh1;
                if (ph == 0) {
                  const float fo = fold_right ? (lw0 + lw1) : lw0;
                  if (own) {
                    O[(int64_t)(lc * 2 + 0) * fwp + t] -= wu * fo;
                    O[(int64_t)(lc * 2 + 1) * fwp + t] -= wl * fo;
                  }
                } else if (!fold_right && t + 1 < kCT && (x + 1) < x_end) {
                  O[(int64_t)(lc * 2 + 0) * fwp + t + 1] -= wu * lw1;
                  O[(int64_t)(lc * 2 + 1) * fwp + t + 1] -= wl * lw1;
                }
              }
            }
          }
          __syncthreads();
        }
        // write the tile: plane A row g (upper), plane B row g+1 (lower)
        for (int e = t; e < cc * n_own; e += kCT) {
          const int c = e / n_own, k = e - c * n_own;  // k-th owned cell <-> thread k+1
          const int xc = xa + k;
          if (xc >= x_end) continue;
          float u = O[(int64_t)(c * 2 + 0) * fwp + k + 1];
          float lw = O[(int64_t)(c * 2 + 1) * fwp + k + 1];
          if (fold_down) { u += lw; lw = 0.f; }
          float* pa = dA + (int64_t)(c_lo + c) * hw + (int64_t)g * gm.w + xc;
          if (first_tile) *pa = u; else *pa += u;
          if (!fold_down) {
            float* pb = dB + (int64_t)(c_lo + c) * hw + (int64_t)(g + 1) * gm.w + xc;
            if (first_tile) *pb = lw; else *pb += lw;
          }
          if (g == 0 && first_tile) dB[(int64_t)(c_lo + c) * hw + xc] = 0.f;  // row 0 of plane B has no producer
        }
      }
      first_tile = false;
    }
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
constexpr size_t kSmemBudget = 56 * 1024;  // per CTA: keeps 3-4 CTAs resident per SM

template <typename T, typename L>
int launch_fwd(const FwdArgs& a0, int n_images, cudaStream_t s) {
  FwdArgs a = a0;
  a.fwp = kCT + 1 + 3;  // fw <= kCT+1; odd-ish pitch keeps the two rows in different banks
  const int C = max_c(&a.src);
  const size_t fixed = (size_t)(2 * a.fwp + kWarps * 2 * kRowBuf) * 4;
  int cc = (int)((kSmemBudget - fixed) / ((size_t)2 * a.fwp * 4));
  if (cc > C) cc = C;
  if (cc < 1) cc = 1;
  a.cc_max = cc;
  const size_t smem = fixed + (size_t)cc * 2 * a.fwp * 4;
  auto k = up_ce_fwd_kernel<T, L>;
  if (smem > 48 * 1024) MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((unsigned)((a.gm.w + kCT - 1) / kCT), (unsigned)a.gm.h, (unsigned)n_images);
  k<<<grid, kCT, smem, s>>>(a);
  MDSEG_LAUNCH_OK();
  return 0;
}

template <typename T, typename L>
int launch_bwd(const BwdArgs& a0, int n_images, cudaStream_t s) {
  BwdArgs a = a0;
  a.fwp = kCT + 1 + 3;
  const int C = max_c(&a.src);
  int cc = (int)(kSmemBudget / ((size_t)(4 * a.fwp + 2 * kWarps) * 4));
  if (cc > C) cc = C;
  if (cc < 1) cc = 1;
  a.cc_max = cc;
  const size_t smem = (size_t)cc * (4 * a.fwp + 2 * kWarps) * 4;
  auto k = up_ce_bwd_kernel<T, L>;
  if (smem > 48 * 1024) MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int n_own = kCT - 1;
  dim3 grid((unsigned)((a.gm.w + n_own - 1) / n_own), (unsigned)a.gm.h, (unsigned)n_images);
  k<<<grid, kCT, smem, s>>>(a);
  MDSEG_LAUNCH_OK();
  return 0;
}

__global__ void add_planes_kernel_f32(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ o,
                                      int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    o[i] = a[i] + b[i];
}
template <typename T>
__global__ void add_planes_kernel(const float* __restrict__ a, const float* __restrict__ b, T* __restrict__ o,
                                  int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    o[i] = from_f32<T>(a[i] + b[i]);
}

}  // namespace
}  // namespace mdseg

extern "C" int mdseg_up_ce_fwd(const mdseg_src_table* src, const int32_t* dataset_ids, const void* labels,
                               int label_dtype, int n_images, int h, int w, int H, int W, int ignore, float* loss_px,
                               float* lse_px, mdseg_ohem_state* states, int32_t* err_flag, void* stream) {
  using namespace mdseg;
  if (int rc = check_src(src, "mdseg_up_ce_fwd")) return rc;
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0 && H > 0 && W > 0 && h <= 65535,
                "mdseg_up_ce_fwd: bad shape");
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(labels && loss_px && lse_px && states && err_flag, "mdseg_up_ce_fwd: null pointer");
  FwdArgs a;
  a.src = *src; a.dataset_ids = dataset_ids; a.labels = labels; a.gm = make_geom(h, w, H, W);
  a.ignore = ignore; a.loss_px = loss_px; a.lse_px = lse_px; a.states = states; a.err_flag = err_flag;
  a.cc_max = 0; a.fwp = 0;
  cudaStream_t s = (cudaStream_t)stream;
  {
    const int rc = up_ce_fwd_warp(a, label_dtype, n_images, s);  // + uint8 labels, W % 16 == 0, cmax ready
    if (rc >= 0) return rc;
  }
  {
    const int rc = up_ce_fwd_tma(a, label_dtype, n_images, s);  // fp32, w % 4 == 0, factor <= 5, cmax workspace
    if (rc >= 0) return rc;
  }
  return with_float_type(src->dtype, "mdseg_up_ce_fwd", "dtype", [&](auto t) {
    return with_int_type(label_dtype, "mdseg_up_ce_fwd", "label dtype", [&](auto l) {
      return launch_fwd<typename decltype(t)::type, typename decltype(l)::type>(a, n_images, s);
    });
  });
}

extern "C" int mdseg_up_ce_bwd(const mdseg_src_table* src, const int32_t* dataset_ids, const void* labels,
                               int label_dtype, int n_images, int h, int w, int H, int W, int ignore,
                               const float* loss_px, const float* lse_px, mdseg_ohem_state* states,
                               const float* grad_out, float grad_scale, const mdseg_src_table* dstA,
                               const mdseg_src_table* dstB, void* stream) {
  using namespace mdseg;
  if (int rc = check_src(src, "mdseg_up_ce_bwd")) return rc;
  if (int rc = check_src(dstA, "mdseg_up_ce_bwd(dstA)")) return rc;
  if (int rc = check_src(dstB, "mdseg_up_ce_bwd(dstB)")) return rc;
  MDSEG_REQUIRE(dstA->dtype == MDSEG_F32 && dstB->dtype == MDSEG_F32, "mdseg_up_ce_bwd: gradient planes must be fp32");
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535 && h > 0 && w > 0 && H > 0 && W > 0 && h <= 65535,
                "mdseg_up_ce_bwd: bad shape");
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(labels && loss_px && lse_px && states, "mdseg_up_ce_bwd: null pointer");
  BwdArgs a;
  a.src = *src; a.dstA = *dstA; a.dstB = *dstB; a.dataset_ids = dataset_ids; a.labels = labels;
  a.gm = make_geom(h, w, H, W); a.ignore = ignore; a.loss_px = loss_px; a.lse_px = lse_px; a.states = states;
  a.grad_out = grad_out; a.grad_scale = grad_scale; a.cc_max = 0; a.fwp = 0;
  cudaStream_t s = (cudaStream_t)stream;
  {
    const int rc = up_ce_bwd_tma(a, label_dtype, n_images, s);
    if (rc >= 0) return rc;
  }
  return with_float_type(src->dtype, "mdseg_up_ce_bwd", "dtype", [&](auto t) {
    return with_int_type(label_dtype, "mdseg_up_ce_bwd", "label dtype", [&](auto l) {
      return launch_bwd<typename decltype(t)::type, typename decltype(l)::type>(a, n_images, s);
    });
  });
}

extern "C" int mdseg_add_planes(const float* a, const float* b, void* out, int out_dtype, int64_t n, void* stream) {
  using namespace mdseg;
  MDSEG_REQUIRE(n >= 0, "mdseg_add_planes: n < 0");
  if (n == 0) return 0;
  MDSEG_REQUIRE(a && b && out, "mdseg_add_planes: null pointer");
  int64_t blocks = ceil_div64(n, 256);
  int64_t cap = (int64_t)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  cudaStream_t s = (cudaStream_t)stream;
  return with_float_type(out_dtype, "mdseg_add_planes", "out_dtype", [&](auto t) {
    using T = typename decltype(t)::type;
    if constexpr (std::is_same_v<T, float>)
      add_planes_kernel_f32<<<(unsigned)blocks, 256, 0, s>>>(a, b, (float*)out, n);
    else
      add_planes_kernel<T><<<(unsigned)blocks, 256, 0, s>>>(a, b, (T*)out, n);
    MDSEG_LAUNCH_OK();
    return 0;
  });
}
