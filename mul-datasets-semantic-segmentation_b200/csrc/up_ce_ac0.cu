// up_ce_ac0.cu — fused bilinear upsample (align_corners=False, power-of-two factors) + per-pixel
// cross-entropy, forward and adjoint.
//
// Reference work replaced (BiSeNet SegmentHead's trailing
//   nn.Upsample(scale_factor=f, mode='bilinear', align_corners=False)
// plus lib/loss/ohem_ce_loss.py:12-34 on its output, and their autograd replay).  ATen writes the
// [N, C, H, W] up-sampled tensor, the CE reads it forward and backward, and the up-sample backward
// scatters into the low-resolution gradient with atomics.  Here only the low-resolution logits are read.
//
// Geometry (ATen area_pixel_compute_source_index, align_corners=False, scale = 1/f exactly):
//   src = max((o + 0.5) / f - 0.5, 0),  i0 = floor(src),  i1 = min(i0 + 1, n_in - 1),  l1 = src - i0.
// For f in {2, 4, 8, 16}, output o = f*i + f/2 + k (k in [0, f)) has i0 = i and l1 = (k + 0.5) / f, an exact
// dyadic fraction, for every i in [-1, n_in - 1] once the corner indices are clamped to [0, n_in - 1]: cell -1
// (the first f/2 outputs, clamped by ATen to l1 = 0 on input 0) and cell n_in - 1 (the last f/2, i1 = i0) have
// both corners on the same input, where the interpolation a + l1 (a - a) returns a exactly.  So every thread
// sees the same constant weights, and the edges only change where the adjoint sends its sums.
//
//  * CTA = one image, one low-res row pair (g, g+1), g in [-1, h-1] (rows clamped), and a band of kT / fy
//    cells [xa - 1, xa + nb - 1) including one left halo cell.  Thread = one label row (Y = fy g + fy/2 + r)
//    of one cell (FX label pixels), constant vertical weight l1h = (r + 0.5) / fy.
//  * The two low-res rows are staged per class chunk in shared memory, pre-multiplied by log2(e).
//  * softmax shift: the bilinear interpolation of the per-corner channel maxima, an upper bound of
//    max_c z_c for non-negative weights: Σ 2^(z - M) needs no online rescale.
//  * backward = adjoint in gather form: per class, the thread sums (p - [c == label])·l0w and ·l1w over its
//    pixels (the four corner sums with its vertical weights) and writes them to a per-thread shared slot;
//    the sums over the cell's rows and the neighbouring cell are then taken in a fixed order.  Plane A
//    receives row g, plane B row g+1; mdseg_add_planes adds them into the source dtype.  No float atomics:
//    the gradient is bit-reproducible.
#include <float.h>

#include "common.cuh"

namespace mdseg {
namespace {

constexpr int kT = 256;                    // threads per CTA: fy label rows x (kT / fy) cells
constexpr int kWarps = kT / 32;
constexpr size_t kSmemBudget = 56 * 1024;  // per CTA: keeps 3-4 CTAs resident per SM

struct Ac0Geom {
  int h, w, H, W;
  int fy;     // H / h
  int nb;     // cells per CTA band, kT / fy, one of them the left halo
  int pitch;  // staged row pitch (>= nb + 1 columns)
  int qp;     // pitch of the backward's per-thread slots (>= nb, bank-conflict free for a warp)
};

struct Ac0Fwd {
  mdseg_src_table src;
  const int32_t* dataset_ids;
  const void* labels;
  Ac0Geom gm;
  int ignore;
  int cc;  // classes per staged chunk
  float* loss_px;
  float* lse_px;
  mdseg_ohem_state* states;
  int* err_flag;
};

struct Ac0Bwd {
  mdseg_src_table src;
  mdseg_src_table dstA, dstB;  // fp32 planes, dense [n_images, C_d, h, w]
  const int32_t* dataset_ids;
  const void* labels;
  Ac0Geom gm;
  int ignore;
  int cc;
  const float* loss_px;
  const float* lse_px;
  mdseg_ohem_state* states;
  const float* grad_out;
  float grad_scale;
};

// Classes [c_lo, c_lo + cc) of low-res rows ytop / ybot, staged columns i <-> xa - 1 + i (clamped to [0, w-1]),
// i < nb + 1, into S[(c * 2 + row) * pitch + i], scaled by log2(e).
template <typename T>
__device__ __forceinline__ void stage_rows(float* __restrict__ S, const T* __restrict__ img, int c_lo, int cc,
                                           int ytop, int ybot, int xa, const Ac0Geom& gm) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t hw = (int64_t)gm.h * gm.w;
  const int ncol = gm.nb + 1;
  for (int cr = warp; cr < cc * 2; cr += kWarps) {
    const int c = cr >> 1;
    const T* row = img + (int64_t)(c_lo + c) * hw + (int64_t)((cr & 1) ? ybot : ytop) * gm.w;
    float* dst = S + (int64_t)cr * gm.pitch;
    for (int i = lane; i < ncol; i += 32) {
      int x = xa - 1 + i;
      x = x < 0 ? 0 : (x > gm.w - 1 ? gm.w - 1 : x);
      dst[i] = to_f32<T>(row[x]) * kLog2e;
    }
  }
}

// cm[row * pitch + i] = log2(e) * max_c src[c][row][column of staged i], over all C classes
template <typename T>
__device__ __forceinline__ void channel_max(float* __restrict__ cm, const float* __restrict__ S, const T* __restrict__ img,
                                            int C, bool staged, int ytop, int ybot, int xa, const Ac0Geom& gm) {
  const int ncol = gm.nb + 1;
  const int64_t hw = (int64_t)gm.h * gm.w;
  for (int e = threadIdx.x; e < 2 * ncol; e += kT) {
    const int row = e / ncol, i = e - row * ncol;
    float m = -FLT_MAX;
    if (staged) {
      for (int c = 0; c < C; ++c) m = fmaxf(m, S[(int64_t)(c * 2 + row) * gm.pitch + i]);
    } else {
      int x = xa - 1 + i;
      x = x < 0 ? 0 : (x > gm.w - 1 ? gm.w - 1 : x);
      const T* p = img + (int64_t)(row ? ybot : ytop) * gm.w + x;
      for (int c = 0; c < C; ++c) m = fmaxf(m, to_f32<T>(p[(int64_t)c * hw]));
      m *= kLog2e;
    }
    cm[row * gm.pitch + i] = m;
  }
}

// horizontal weight of pixel k of a cell: (k + 0.5) / FX, exact
template <int FX>
__device__ __forceinline__ constexpr float l1w_of(int k) {
  return ((float)k + 0.5f) / (float)FX;
}

// ---------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------
// explicit register caps: under __launch_bounds__(kT) alone ptxas spills a few words of the set-up at FX = 2, 4
template <typename T, typename L, int FX>
__global__ void __maxnreg__(FX >= 8 ? 80 : 64)
up_ce_ac0_fwd_kernel(const Ac0Fwd a) {
  extern __shared__ float smem[];
  const Ac0Geom& gm = a.gm;
  const int t = threadIdx.x, b = blockIdx.z, g = (int)blockIdx.y - 1;
  const int xa = blockIdx.x * (gm.nb - 1);  // first owned cell of the band
  const int cl = t / gm.fy, r = t - cl * gm.fy;
  const int x = xa - 1 + cl;                // this thread's cell
  const int Y = gm.fy * g + gm.fy / 2 + r;  // this thread's label row
  const int X0 = FX * x + FX / 2;           // first label column of the cell
  // the band's halo cell belongs to the previous band, except cell -1 (the first FX/2 columns)
  const bool mine = (x >= xa || x == -1) && x < gm.w && Y >= 0 && Y < gm.H;
  const int k_lo = X0 < 0 ? -X0 : 0;
  const int k_hi = (gm.W - X0) < FX ? (gm.W - X0) : FX;
  const L* labels = (const L*)a.labels;
  const int64_t rowbase = ((int64_t)b * gm.H + Y) * gm.W + X0;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;

  unsigned n_valid = 0, n_hard = 0, n_px = 0;
  double sum_hard = 0.0;
  int err = 0;

  if (d < 0 || d >= a.src.n_datasets) {
    // image outside every dataset: not part of the loss vector (sentinel -1), but its labels still count in
    // n_min (ohem_ce_loss.py:25 counts all labels)
    if (mine)
      for (int k = k_lo; k < k_hi; ++k) {
        a.loss_px[rowbase + k] = -1.0f;
        a.lse_px[rowbase + k] = 0.f;
        n_valid += (load_label<L>(labels, rowbase + k) != a.ignore) ? 1u : 0u;
      }
    if (t == 0 && blockIdx.x == 0 && blockIdx.y == 0) atomicOr(a.err_flag, MDSEG_ERR_DATASET_ID);
    block_accumulate_stats(a.states, n_valid, 0u, 0.0, 0u);
    return;
  }
  const int C = a.src.C[d];
  const T* img = (const T*)a.src.base[d] + (int64_t)b * a.src.image_stride[d];
  mdseg_ohem_state* st = a.states + (a.src.seg_per_dataset ? d : 0);
  const float thresh = st->thresh;

  const int ytop = g < 0 ? 0 : g;
  const int ybot = (g + 1) > gm.h - 1 ? gm.h - 1 : g + 1;
  const int pitch = gm.pitch;
  float* cm = smem;                // [2][pitch]
  float* S = smem + 2 * pitch;     // [cc][2][pitch]
  const bool single_chunk = C <= a.cc;
  if (single_chunk) {
    stage_rows<T>(S, img, 0, C, ytop, ybot, xa, gm);
    __syncthreads();
  }
  channel_max<T>(cm, S, img, C, single_chunk, ytop, ybot, xa, gm);
  __syncthreads();

  const float l1h = ((float)r + 0.5f) / (float)gm.fy;
  const float m0 = cm[cl] + l1h * (cm[pitch + cl] - cm[cl]);
  const float m1 = cm[cl + 1] + l1h * (cm[pitch + cl + 1] - cm[cl + 1]);

  int lab[FX];
  float s[FX], tl[FX];  // Σ_c 2^(z_c - M) and z_label - M, per pixel (log2 units)
#pragma unroll
  for (int k = 0; k < FX; ++k) {
    lab[k] = (mine && k >= k_lo && k < k_hi) ? load_label<L>(labels, rowbase + k) : a.ignore;
    s[k] = 0.f;
    tl[k] = 0.f;
  }

  for (int c_lo = 0; c_lo < C; c_lo += a.cc) {
    const int cc = (C - c_lo) < a.cc ? (C - c_lo) : a.cc;
    if (!single_chunk) {
      __syncthreads();
      stage_rows<T>(S, img, c_lo, cc, ytop, ybot, xa, gm);
      __syncthreads();
    }
    const float* Sp = S + cl;
#pragma unroll 2
    for (int c = 0; c < cc; ++c) {
      const float v00 = Sp[0], v01 = Sp[1], v10 = Sp[pitch], v11 = Sp[pitch + 1];
      Sp += 2 * pitch;
      const float e0 = (v00 + l1h * (v10 - v00)) - m0;
      const float e1 = (v01 + l1h * (v11 - v01)) - m1;
      const float dd = e1 - e0;
#pragma unroll
      for (int k = 0; k < FX; ++k) s[k] += ex2_approx(fmaf(l1w_of<FX>(k), dd, e0));
    }
    // the label class's term, with the arithmetic of the sum above
#pragma unroll
    for (int k = 0; k < FX; ++k) {
      const unsigned lc = (unsigned)(lab[k] - c_lo);
      if (lab[k] != a.ignore && lc < (unsigned)cc) {
        const float* q = S + (int64_t)lc * 2 * pitch + cl;
        const float e0 = (q[0] + l1h * (q[pitch] - q[0])) - m0;
        const float e1 = (q[1] + l1h * (q[pitch + 1] - q[1])) - m1;
        tl[k] = fmaf(l1w_of<FX>(k), e1 - e0, e0);
      }
    }
  }

  if (mine) {
#pragma unroll
    for (int k = 0; k < FX; ++k) {
      if (k >= k_lo && k < k_hi) {
        const float ls2 = log2f(s[k]);
        const float M = fmaf(l1w_of<FX>(k), m1 - m0, m0);
        const bool ign = lab[k] == a.ignore;
        const bool ok = (unsigned)lab[k] < (unsigned)C;
        if (!ign && !ok) err |= MDSEG_ERR_LABEL_RANGE;
        const float l = (ok && !ign) ? (ls2 - tl[k]) * kLn2 : 0.f;
        a.loss_px[rowbase + k] = l;
        a.lse_px[rowbase + k] = (M + ls2) * kLn2;
        n_valid += (ok && !ign) ? 1u : 0u;
        if (l > thresh) { ++n_hard; sum_hard += (double)l; }
        ++n_px;
      }
    }
  }
  if (err) atomicOr(a.err_flag, err);
  block_accumulate_stats(st, n_valid, n_hard, sum_hard, n_px);
}

// ---------------------------------------------------------------------------
// backward (adjoint, gather form)
// ---------------------------------------------------------------------------
struct SelW {
  float thresh, kth, w;
  unsigned mode;
};
// Membership in S is a pure function of the stored loss (mdseg_ohem_select demotes the ties that missed the
// top-k quota to just below kth).
__device__ __forceinline__ bool selected(const SelW& p, float loss) {
  return p.mode == 0 ? (loss > p.thresh) : (loss >= p.kth);
}

template <typename T, typename L, int FX>
__global__ void __launch_bounds__(kT)
up_ce_ac0_bwd_kernel(const Ac0Bwd a) {
  extern __shared__ float smem[];
  const Ac0Geom& gm = a.gm;
  const int t = threadIdx.x, b = blockIdx.z, g = (int)blockIdx.y - 1;
  const int d = a.dataset_ids ? a.dataset_ids[b] : 0;
  if (d < 0 || d >= a.src.n_datasets) return;  // no gradient rows for this image
  const int C = a.src.C[d];
  const T* img = (const T*)a.src.base[d] + (int64_t)b * a.src.image_stride[d];
  float* dA = (float*)a.dstA.base[d] + (int64_t)b * a.dstA.image_stride[d];
  float* dB = (float*)a.dstB.base[d] + (int64_t)b * a.dstB.image_stride[d];
  const mdseg_ohem_state* st = a.states + (a.src.seg_per_dataset ? d : 0);
  SelW sp;
  sp.thresh = st->thresh; sp.kth = st->kth; sp.mode = st->mode;
  sp.w = (a.grad_out ? a.grad_out[a.src.seg_per_dataset ? d : 0] : 1.f) * a.grad_scale * st->inv_n_sel;

  const int n_own = gm.nb - 1;
  const int xa = blockIdx.x * n_own;
  const int fy = gm.fy;
  const int cl = t / fy, r = t - cl * fy;
  const int x = xa - 1 + cl;
  const int Y = fy * g + fy / 2 + r;
  const int X0 = FX * x + FX / 2;
  // every cell of the band is computed (the halo's right-corner sums belong to column xa)
  const bool rows_ok = x < gm.w && Y >= 0 && Y < gm.H;
  const int k_lo = X0 < 0 ? -X0 : 0;
  const int k_hi = (gm.W - X0) < FX ? (gm.W - X0) : FX;
  const L* labels = (const L*)a.labels;
  const int64_t rowbase = ((int64_t)b * gm.H + Y) * gm.W + X0;

  // unselected / ignored / outside pixels: lse = +inf makes their softmax term 0; lab = -1 drops the label term
  float lse2[FX];
  int lab[FX];
#pragma unroll
  for (int k = 0; k < FX; ++k) {
    lse2[k] = __int_as_float(0x7f800000);
    lab[k] = -1;
    if (rows_ok && k >= k_lo && k < k_hi) {
      const int lb = load_label<L>(labels, rowbase + k);
      if (lb != a.ignore && (unsigned)lb < (unsigned)C && selected(sp, a.loss_px[rowbase + k])) {
        lse2[k] = a.lse_px[rowbase + k] * kLog2e;
        lab[k] = lb;
      }
    }
  }
  const float l1h = ((float)r + 0.5f) / (float)fy;
  const float wu = sp.w * (1.f - l1h), wl = sp.w * l1h;  // upper / lower row weights times 1/|S|

  const int ytop = g < 0 ? 0 : g;
  const int ybot = (g + 1) > gm.h - 1 ? gm.h - 1 : g + 1;
  const int pitch = gm.pitch, qp = gm.qp;
  float* S = smem;                                  // [cc][2][pitch]
  float* Q = smem + (int64_t)a.cc * 2 * pitch;      // [cc][4][fy][qp]: upper x0, upper x1, lower x0, lower x1
  const int64_t hw = (int64_t)gm.h * gm.w;
  float* slot = Q + (int64_t)r * qp + cl;
  const int64_t qcls = (int64_t)4 * fy * qp, qq = (int64_t)fy * qp;

  for (int c_lo = 0; c_lo < C; c_lo += a.cc) {
    const int cc = (C - c_lo) < a.cc ? (C - c_lo) : a.cc;
    __syncthreads();
    stage_rows<T>(S, img, c_lo, cc, ytop, ybot, xa, gm);
    __syncthreads();
    const float* Sp = S + cl;
    for (int c = 0; c < cc; ++c) {
      const float v00 = Sp[0], v01 = Sp[1], v10 = Sp[pitch], v11 = Sp[pitch + 1];
      Sp += 2 * pitch;
      const float c0 = v00 + l1h * (v10 - v00);
      const float dd = (v01 + l1h * (v11 - v01)) - c0;
      float a0 = 0.f, a1 = 0.f;
#pragma unroll
      for (int k = 0; k < FX; ++k) {
        // p - [c == label] per pixel: for an easy pixel p - 1 is small, and subtracting after the sum would cancel
        float e = ex2_approx(fmaf(l1w_of<FX>(k), dd, c0) - lse2[k]);
        if (lab[k] == c_lo + c) e -= 1.f;
        a0 = fmaf(1.f - l1w_of<FX>(k), e, a0);
        a1 = fmaf(l1w_of<FX>(k), e, a1);
      }
      float* q = slot + c * qcls;
      q[0] = wu * a0;
      q[qq] = wu * a1;
      q[2 * qq] = wl * a0;
      q[3 * qq] = wl * a1;
    }
    __syncthreads();
    // column xo = xa + j gathers the left corners of its own cell (slot j + 1) and the right corners of the
    // cell to its left (slot j); cell -1 has both corners on column 0, cell w - 1 both on column w - 1
    for (int e = t; e < cc * n_own; e += kT) {
      const int c = e / n_own, j = e - c * n_own;
      const int xo = xa + j;
      if (xo >= gm.w) continue;
      const float* qc = Q + c * qcls;
      float up = 0.f, lo = 0.f;
      for (int rr = 0; rr < fy; ++rr) {
        const float* q = qc + (int64_t)rr * qp;
        float u = q[j + 1] + q[qq + j];
        float l = q[2 * qq + j + 1] + q[3 * qq + j];
        if (xo == 0) { u += q[j]; l += q[2 * qq + j]; }
        if (xo == gm.w - 1) { u += q[qq + j + 1]; l += q[3 * qq + j + 1]; }
        up += u;
        lo += l;
      }
      const int64_t o = (int64_t)(c_lo + c) * hw + xo;
      if (g < 0) {
        dB[o] = up + lo;  // rows -1 and 0 are both low-res row 0
      } else if (g == gm.h - 1) {
        dA[o + (int64_t)g * gm.w] = up + lo;  // rows h-1 and h are both low-res row h-1
      } else {
        dA[o + (int64_t)g * gm.w] = up;
        dB[o + (int64_t)(g + 1) * gm.w] = lo;
      }
    }
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
bool pow2_factor(int f) { return f == 2 || f == 4 || f == 8 || f == 16; }

// The geometry these kernels take: H = fy h and W = fx w with fy, fx in {2, 4, 8, 16}.
int make_geom(const char* who, int h, int w, int H, int W, Ac0Geom* gm, int* fx) {
  MDSEG_REQUIRE(h > 0 && w > 0 && H > 0 && W > 0 && h <= 65534, "%s: bad shape", who);
  MDSEG_REQUIRE(H % h == 0 && W % w == 0 && pow2_factor(H / h) && pow2_factor(W / w),
                "%s: align_corners=False up-sampling takes factors 2, 4, 8 or 16 per axis (H = f h, W = f w); "
                "got %dx%d -> %dx%d",
                who, h, w, H, W);
  gm->h = h; gm->w = w; gm->H = H; gm->W = W;
  gm->fy = H / h;
  gm->nb = kT / gm->fy;
  gm->pitch = gm->nb + 1;
  // smallest slot pitch >= nb under which the 32 lanes of a warp (fy rows x 32/fy cells) hit 32 banks
  for (int qp = gm->nb;; ++qp) {
    unsigned used = 0;
    for (int lane = 0; lane < 32; ++lane) used |= 1u << (((lane % gm->fy) * qp + lane / gm->fy) & 31);
    if (used == 0xffffffffu) { gm->qp = qp; break; }
  }
  *fx = W / w;
  return 0;
}

template <typename T, typename L, int FX>
int launch_fwd(const Ac0Fwd& a0, int n_images, cudaStream_t s) {
  Ac0Fwd a = a0;
  const size_t per_class = (size_t)2 * a.gm.pitch * 4;
  const size_t fixed = per_class;  // channel maxima
  int cc = (int)((kSmemBudget - fixed) / per_class);
  const int C = max_c(&a.src);
  a.cc = cc > C ? C : cc;
  const size_t smem = fixed + (size_t)a.cc * per_class;
  auto k = up_ce_ac0_fwd_kernel<T, L, FX>;
  if (smem > 48 * 1024) MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int n_own = a.gm.nb - 1;
  dim3 grid((unsigned)((a.gm.w + n_own - 1) / n_own), (unsigned)(a.gm.h + 1), (unsigned)n_images);
  k<<<grid, kT, smem, s>>>(a);
  MDSEG_LAUNCH_OK();
  return 0;
}

template <typename T, typename L, int FX>
int launch_bwd(const Ac0Bwd& a0, int n_images, cudaStream_t s) {
  Ac0Bwd a = a0;
  const size_t per_class = ((size_t)2 * a.gm.pitch + (size_t)4 * a.gm.fy * a.gm.qp) * 4;
  const int cc = (int)(kSmemBudget / per_class);
  const int C = max_c(&a.src);
  a.cc = cc > C ? C : cc;
  const size_t smem = (size_t)a.cc * per_class;
  auto k = up_ce_ac0_bwd_kernel<T, L, FX>;
  if (smem > 48 * 1024) MDSEG_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int n_own = a.gm.nb - 1;
  dim3 grid((unsigned)((a.gm.w + n_own - 1) / n_own), (unsigned)(a.gm.h + 1), (unsigned)n_images);
  k<<<grid, kT, smem, s>>>(a);
  MDSEG_LAUNCH_OK();
  return 0;
}

// source dtype x label dtype x horizontal factor
template <bool kFwd, typename Args>
int run(const Args& a, int dtype, int label_dtype, int fx, int n_images, cudaStream_t s, const char* who) {
  return with_float_type(dtype, who, "dtype", [&](auto t) {
    return with_int_type(label_dtype, who, "label dtype", [&](auto l) -> int {
      using T = typename decltype(t)::type;
      using L = typename decltype(l)::type;
      switch (fx) {
#define MDSEG_AC0_FX(F) \
  case F:               \
    if constexpr (kFwd) return launch_fwd<T, L, F>(a, n_images, s); else return launch_bwd<T, L, F>(a, n_images, s);
        MDSEG_AC0_FX(2) MDSEG_AC0_FX(4) MDSEG_AC0_FX(8) MDSEG_AC0_FX(16)
#undef MDSEG_AC0_FX
      }
      return 2;
    });
  });
}

}  // namespace
}  // namespace mdseg

extern "C" int mdseg_up_ce_fwd_ac0(const mdseg_src_table* src, const int32_t* dataset_ids, const void* labels,
                                   int label_dtype, int n_images, int h, int w, int H, int W, int ignore,
                                   float* loss_px, float* lse_px, mdseg_ohem_state* states, int32_t* err_flag,
                                   void* stream) {
  using namespace mdseg;
  static const char* who = "mdseg_up_ce_fwd_ac0";
  Ac0Fwd a;
  int fx = 0;
  if (int rc = make_geom(who, h, w, H, W, &a.gm, &fx)) return rc;
  if (int rc = check_src(src, who)) return rc;
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535, "%s: bad image count %d", who, n_images);
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(labels && loss_px && lse_px && states && err_flag, "%s: null pointer", who);
  a.src = *src; a.dataset_ids = dataset_ids; a.labels = labels; a.ignore = ignore; a.cc = 0;
  a.loss_px = loss_px; a.lse_px = lse_px; a.states = states; a.err_flag = err_flag;
  return run<true>(a, src->dtype, label_dtype, fx, n_images, (cudaStream_t)stream, who);
}

extern "C" size_t mdseg_up_ce_bwd_ac0_workspace_bytes(const mdseg_src_table* src, int n_images, int h, int w, int H,
                                                      int W) {
  using namespace mdseg;
  if (!src_count_ok(src) || n_images <= 0 || h <= 0 || w <= 0) return 256;
  (void)H; (void)W;
  return two_plane_bytes(src, n_images, h, w);
}

extern "C" int mdseg_up_ce_bwd_ac0(const mdseg_src_table* src, const int32_t* dataset_ids, const void* labels,
                                   int label_dtype, int n_images, int h, int w, int H, int W, int ignore,
                                   const float* loss_px, const float* lse_px, mdseg_ohem_state* states,
                                   const float* grad_out, float grad_scale, const mdseg_src_table* dst,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  using namespace mdseg;
  static const char* who = "mdseg_up_ce_bwd_ac0";
  Ac0Bwd a;
  int fx = 0;
  if (int rc = make_geom(who, h, w, H, W, &a.gm, &fx)) return rc;
  if (int rc = check_src(src, who)) return rc;
  MDSEG_REQUIRE(dst && dst->n_datasets == src->n_datasets && is_float_dtype(dst->dtype),
                "%s: bad destination table", who);
  const int64_t hw = (int64_t)h * w;
  for (int i = 0; i < src->n_datasets; ++i)
    MDSEG_REQUIRE(dst->base[i] && dst->C[i] == src->C[i] && dst->image_stride[i] == (long long)src->C[i] * hw,
                  "%s: destination %d must be a dense [n_images, C, h, w] tensor", who, i);
  MDSEG_REQUIRE(n_images >= 0 && n_images <= 65535, "%s: bad image count %d", who, n_images);
  if (n_images == 0) return 0;
  MDSEG_REQUIRE(labels && loss_px && lse_px && states && workspace, "%s: null pointer", who);
  MDSEG_REQUIRE(workspace_bytes >= mdseg_up_ce_bwd_ac0_workspace_bytes(src, n_images, h, w, H, W),
                "%s: workspace too small", who);
  cudaStream_t s = (cudaStream_t)stream;
  a.src = *src; a.dataset_ids = dataset_ids; a.labels = labels; a.ignore = ignore;
  a.cc = 0; a.loss_px = loss_px; a.lse_px = lse_px; a.states = states; a.grad_out = grad_out;
  a.grad_scale = grad_scale;
  // the kernel writes both planes of every image of a valid dataset id; with several datasets (or ids) the planes
  // of the other heads' images are zero, so the sum writes exact zeros there
  const bool zero = dataset_ids || src->n_datasets > 1;
  return two_plane_adjoint(who, src, dst, n_images, h, w, workspace, zero, s,
                           [&](const mdseg_src_table& dA, const mdseg_src_table& dB) {
                             a.dstA = dA; a.dstB = dB;
                             return run<false>(a, src->dtype, label_dtype, fx, n_images, s, who);
                           });
}
