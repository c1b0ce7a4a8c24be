// The per-pixel loss evaluated straight from the network's LOW-RES logits (SURVEY 8f-1).
//
// The reference network ends with  logits = F.interpolate(sem_logits, size=(H,W), mode="bilinear",
// align_corners=False)  (networks/deeplab_v3.py:154-160) and hands the [B,K,H,W] tensor to the loss; autograd later
// pushes a [B,K,H,W] gradient back through the same up-sample.  Here the up-sample, every per-pixel loss term of
// pixel_loss.cu (same pixel_terms(): weighted / plain / unbiased CE, score, seen-detector focal term, distill mask,
// arg-max) and the ADJOINT of the up-sample run in one kernel: it reads sem_logits [B,K,lh,lw] (2.7 MB at VOC
// sizes instead of 264 MB), never materialises a full-resolution logit or gradient, and writes d(loss)/d(sem_logits).
// HBM traffic per pixel drops from 2*K*s + 17 bytes to 17 bytes (label, arg-max, mask): the kernel is bound by
// instruction issue / MUFU, not by HBM.
//
// Work split: a thread owns the SX = W/lw consecutive pixels [SX*j, SX*j+SX) of one image row.  Inside that span the
// up-sampled logit of channel c is  v_j + s_i * D  with s_i = (i+0.5)/SX - 0.5 and D = v_j - v_{j-1} (left half,
// s_i < 0) or v_{j+1} - v_j (right half) -- v_* are the low-res columns interpolated in y for this row, columns
// clamped at the image border exactly like ATen's half-pixel rule.  Any other width (EXACT = false: lw = ceil(W / SX),
// what a backbone with padded stride-2 convolutions returns for an input that is not a multiple of its output
// stride): thread j owns the pixels whose half-pixel source column rounds to j, at most SX of them; s_i = src_x - j
// is a runtime per-pixel value and pixels past the span are predicated off.  The channel loop is the OUTER loop (any
// K, no shared-memory logit tile): pass 1a max / arg-max, pass 1b exponent sums, per-pixel terms, pass 2 gradients, which
// are reduced over the SX pixels in registers (sum g, sum s_i g per half) before they touch memory: three plain
// shared-memory stores per (thread, channel); after every chunk of 8 channels the CTA sums its rows with their
// y-weights and sends one global fp32 RED per low-res cell (shared-memory fp32 atomics are CAS loops on sm_100).
// The per-pixel stage (pixel_terms, seen heads) runs as a rolled loop over dynamically indexed copies of the
// per-pixel statistics, so its code exists once instead of SX times.
//
// PSEUDO = true is the arg-max-only instantiation behind bacs_pseudo_label_lowres (csrc/pseudo.cu): `labels` and `preds`
// are the same tensor; a thread reads its labels, runs pass 1a when one of them is 0, writes the arg-max at exactly
// those pixels and returns -- the pseudo label is bit for bit the `preds` of the loss kernel at the same sem_logits.
#pragma once
#include "pixel_common.cuh"

namespace bacs {

struct alignas(16) LowresParams {
  bacs_pixel_args a;     // logits = sem_logits [B,K,lh,lw]; dlogits unused by the kernel (see g32)
  float* g32;            // [B,K,lh,lw] fp32 gradient accumulator (zeroed by the caller) or nullptr
  int lh, lw;            // low-res logit size; W == lw * SX (EXACT) or lw == ceil(W / SX)
  int R;                 // image rows per CTA (R * lw <= 256 threads)
  int groups_per_image;  // ceil(H / R)
  int nsrc_max;          // source rows staged per CTA (shared-memory sizing)
  float hy;              // half-pixel scale lh / H
  float inv_n;           // 1 / (B*H*W)
  float sy, sx;          // align_corners=True scales of the seen heads
  double* partials;      // [grid, BACS_NACC]
  float hx;              // half-pixel scale lw / W (EXACT = false)
};

constexpr int kLowresThreads = 256;
constexpr int kLowresChunk = 8;   // channels per gradient-reduction round
constexpr int kLowresMaxSrc = 8;  // source rows a row group may touch (the host halves R until it holds)
constexpr size_t kLowresMaxSmem = (size_t)200 * 1024;  // dynamic shared memory of one CTA (two CTAs per SM)

struct LowresPlan {
  int SX, R, groups, nsrc_max, grid;
  bool exact;  // W == SX * lw: the instantiation with compile-time pixel offsets
  size_t smem, part_bytes, g32_bytes;
};
// The plan of a launch of pixel_lowres_kernel for `a` at low-res size lh x lw; false when the geometry is not served
// (pixel_loss.cu).  bacs_pseudo_label_lowres accepts exactly what bacs_pixel_loss_lowres accepts without `z`.
bool make_lowres_plan(const bacs_pixel_args& a, int lh, int lw, LowresPlan* plan);

// half-pixel source column of output pixel x (lerp_half_pixel's src, op by op) and the column it rounds to
__device__ __forceinline__ float lowres_src(int x, float scale) {
  const float s = __fsub_rn(__fmul_rn(scale, __fadd_rn((float)x, 0.5f)), 0.5f);
  return s < 0.f ? 0.f : s;
}
__device__ __forceinline__ int lowres_owner(int x, float scale) { return (int)__fadd_rn(lowres_src(x, scale), 0.5f); }
// first pixel of column j's span (W for j == lw).  The owner is monotone in x, so the spans [start(j), start(j+1))
// cover the row once; host_span_start (pixel_loss.cu) is the host copy the plan checks the span lengths with.
__device__ __forceinline__ int lowres_span_start(int j, int lw, int W, float scale) {
  if (j >= lw) return W;
  int x = (int)((int64_t)j * W / lw);
  while (x > 0 && lowres_owner(x - 1, scale) >= j) --x;
  while (x < W && lowres_owner(x, scale) < j) ++x;
  return x;
}

template <int SX, bool EXACT, bool PSEUDO = false>
__global__ void __launch_bounds__(kLowresThreads, 2) pixel_lowres_kernel(const __grid_constant__ LowresParams p) {
  extern __shared__ __align__(16) unsigned char lr_smem[];
  __shared__ float red_scratch[kLowresThreads / 32][BACS_NACC];
  __shared__ float s_norm_sh;
  const bacs_pixel_args& a = p.a;
  constexpr int CH = kLowresChunk;
  const int K = a.K, lh = p.lh, lw = p.lw, LWP = lw + 2, R = p.R;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int b = (int)blockIdx.x / p.groups_per_image;
  const int y0 = ((int)blockIdx.x - b * p.groups_per_image) * R;
  const int rows = min(R, a.H - y0);
  const int64_t HW = (int64_t)a.H * a.W;
  const int old_cl = min(max(a.old_cl, 0), K);
  const bool have_seen = (a.z != nullptr) || (a.seen_max != nullptr);

  // source rows of this row group (ATen half-pixel rule, area_pixel_compute_source_index)
  const Lerp lfirst = lerp_half_pixel(y0, lh, p.hy), llast = lerp_half_pixel(y0 + rows - 1, lh, p.hy);
  const int base = lfirst.i0, nsrc = llast.i1 - base + 1;

  float* src = reinterpret_cast<float*>(lr_smem);          // [nsrc_max][K][lw + 2]  (columns clamped into the pads)
  float* planes = src + (size_t)p.nsrc_max * K * LWP;      // [3][R][CH][lw]         per-row gradient contributions
  float* wrow = planes + (size_t)3 * R * CH * lw;          // [nsrc_max][R]          y-weight of row r on source row n
  float* zr = wrow + (size_t)p.nsrc_max * R;               // [R][T][w]              seen heads, interpolated in y
  float* gacc = zr + (a.z ? (size_t)R * a.T * a.w : 0);    // [R][w + 1]             focal gradient rows
  const size_t plane_sz = (size_t)R * CH * lw;

  // ---- stage ------------------------------------------------------------------------------------------------------
  {
    const int64_t img = (int64_t)b * K * lh * lw;
    for (int t = wid; t < nsrc * K; t += kLowresThreads / 32) {
      const int n = t / K, c = t - n * K;
      const int64_t off = img + ((int64_t)c * lh + base + n) * lw;
      float* row = src + (size_t)t * LWP;
      for (int col = lane; col < lw; col += 32) {
        float v;
        if (a.dtype == BACS_F32) v = __ldg(reinterpret_cast<const float*>(a.logits) + off + col);
        else if (a.dtype == BACS_BF16) v = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(a.logits)[off + col]);
        else v = __half2float(reinterpret_cast<const __half*>(a.logits)[off + col]);
        row[col + 1] = v;
        if (col == 0) row[0] = v;
        if (col == lw - 1) row[lw + 1] = v;
      }
    }
    for (int idx = tid; idx < p.nsrc_max * R; idx += kLowresThreads) {
      const int n = idx / R, rr = idx - n * R;
      float wv = 0.f;
      if (rr < rows) {
        const Lerp ly = lerp_half_pixel(y0 + rr, lh, p.hy);
        if (ly.i0 - base == n) wv += 1.f - ly.w1;
        if (ly.i1 - base == n) wv += ly.w1;
      }
      wrow[idx] = wv;
    }
    if (a.z) {
      const float* zb = a.z + (int64_t)b * a.T * a.h * a.w;
      for (int t2 = wid; t2 < rows * a.T; t2 += kLowresThreads / 32) {
        const int rr = t2 / a.T, t = t2 - rr * a.T;
        const Lerp ly = lerp_align_corners(y0 + rr, a.h, p.sy);
        const float* zt = zb + (int64_t)t * a.h * a.w;
        for (int jj = lane; jj < a.w; jj += 32)
          zr[(size_t)t2 * a.w + jj] = __fadd_rn(__fmul_rn(1.f - ly.w1, __ldg(zt + ly.i0 * a.w + jj)),
                                               __fmul_rn(ly.w1, __ldg(zt + ly.i1 * a.w + jj)));
      }
      if (a.gz)
        for (int idx = tid; idx < R * (a.w + 1); idx += kLowresThreads) gacc[idx] = 0.f;
    }
    if (tid == 0) s_norm_sh = 0.f;
  }
  __syncthreads();
  // CE-type modes: gradient normaliser from the label histogram (device-side, no host sync)
  if (tid < 32 && a.mode != BACS_PIX_WEIGHTED_CE && p.g32 != nullptr) {
    double s = 0.0;
    for (int c = tid; c < K && c < 256; c += 32)
      if (c != a.ignore_index)
        s += (double)a.hist[c] * ((a.mode == BACS_PIX_CE && a.class_w) ? (double)a.class_w[c] : 1.0);
    s = warp_sum(s);
    if (tid == 0) s_norm_sh = s > 0.0 ? (float)(1.0 / s) : 0.f;
  }
  __syncthreads();
  const float s_norm = s_norm_sh;

  float acc[BACS_NACC];
#pragma unroll
  for (int i = 0; i < BACS_NACC; ++i) acc[i] = 0.f;

  const int r = tid / lw, j = tid - r * lw;
  const bool active = r < rows;
  constexpr float kInvSX = 1.f / (float)SX;
  // the thread's pixels of its image row: [xs, xs + npx); sxr[i] = src_x - j of pixel i (0 past the span)
  int xs = SX * j, npx = SX;
  float sxr[SX];
  if constexpr (!EXACT) {
    xs = lowres_span_start(j, lw, a.W, p.hx);
    npx = lowres_span_start(j + 1, lw, a.W, p.hx) - xs;
#pragma unroll
    for (int i = 0; i < SX; ++i) sxr[i] = i < npx ? lowres_src(xs + i, p.hx) - (float)j : 0.f;
  }
#define BACS_LR_S(i) (EXACT ? (((float)(i) + 0.5f) * kInvSX - 0.5f) : sxr[i])
#define BACS_LR_LEFT(i) (EXACT ? (i) < SX / 2 : sxr[i] < 0.f)

  // per-thread state that lives from the forward passes to the gradient pass
  F2 nm2[SX / 2], cg1p[SX / 2], cg2p[SX / 2];  // pixel pairs (2i, 2i+1) as packed fp32 (FFMA2 / FMUL2 / FADD2)
  uint32_t ypk[SX / 4];
  float G0 = 0.f, GL0 = 0.f, GR0 = 0.f;
  int ymin = 256, ymax = -1;
  float ty = 0.f, wy0 = 0.f;
  const float* s0 = src;
  const float* s1 = src;
  // the row-interpolated low-res columns of one channel as (v_j, v_j - v_{j-1}, v_{j+1} - v_j)
  auto trio = [&](int c, float& vj, float& dl, float& dr) {
    const float* q0 = s0 + c * LWP;
    const float* q1 = s1 + c * LWP;
    const float vl = fmaf(ty, q1[0], wy0 * q0[0]);
    vj = fmaf(ty, q1[1], wy0 * q0[1]);
    const float vr = fmaf(ty, q1[2], wy0 * q0[2]);
    dl = vj - vl;
    dr = vr - vj;
  };

  if (active) {
    const int Y = y0 + r;
    const Lerp ly = lerp_half_pixel(Y, lh, p.hy);
    ty = ly.w1;
    wy0 = 1.f - ly.w1;
    s0 = src + (size_t)(ly.i0 - base) * K * LWP + j;  // columns j-1, j, j+1 at [0], [1], [2]
    s1 = src + (size_t)(ly.i1 - base) * K * LWP + j;
    const int64_t pix0 = (int64_t)b * HW + (int64_t)Y * a.W + (EXACT ? (int64_t)SX * j : (int64_t)xs);

    // ---- labels: SX int64 -> one byte each (255 = ignored / invalid) ----------------------------------------------
    uint32_t bg = 0;  // PSEUDO: bit i set where pixel i is labelled 0
    if constexpr (PSEUDO) {
      const int64_t* lp = a.labels + pix0;
      if (EXACT && (reinterpret_cast<uintptr_t>(lp) & 15) == 0) {
#pragma unroll
        for (int i = 0; i < SX; i += 2) {
          const longlong2 v = *reinterpret_cast<const longlong2*>(lp + i);
          bg |= ((uint32_t)(v.x == 0) << i) | ((uint32_t)(v.y == 0) << (i + 1));
        }
      } else {
#pragma unroll
        for (int i = 0; i < SX; ++i)
          if (EXACT || i < npx) bg |= (uint32_t)(lp[i] == 0) << i;
      }
      if (bg == 0) return;  // no pixel to rewrite (no barrier follows in this instantiation)
    } else if constexpr (!EXACT) {  // scalar loads; pixels past the span read as ignored
      const int64_t* lp = a.labels + pix0;
#pragma unroll
      for (int q = 0; q < SX / 4; ++q) ypk[q] = 0;
#pragma unroll
      for (int i = 0; i < SX; ++i) {
        uint32_t y8 = 255u;
        if (i < npx) {
          const long long l = __ldg(lp + i);
          if (l == a.ignore_index) {
          } else if (l >= 0 && l < K) {
            y8 = (uint32_t)l;
            ymin = min(ymin, (int)l);
            ymax = max(ymax, (int)l);
          } else {
            acc[BACS_ACC_INVALID] += 1.f;
          }
        }
        ypk[i >> 2] |= y8 << (8 * (i & 3));
      }
    } else {
      const int64_t* lp = a.labels + pix0;
#pragma unroll
      for (int q = 0; q < SX / 4; ++q) ypk[q] = 0;
      const bool vec = (reinterpret_cast<uintptr_t>(lp) & 15) == 0;
#pragma unroll
      for (int i = 0; i < SX; i += 2) {
        long long l0, l1;
        if (vec) {
          const longlong2 v = __ldg(reinterpret_cast<const longlong2*>(lp + i));
          l0 = v.x;
          l1 = v.y;
        } else {
          l0 = __ldg(lp + i);
          l1 = __ldg(lp + i + 1);
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const long long l = h ? l1 : l0;
          uint32_t y8 = 255u;
          if (l == a.ignore_index) {
          } else if (l >= 0 && l < K) {
            y8 = (uint32_t)l;
            ymin = min(ymin, (int)l);
            ymax = max(ymax, (int)l);
          } else {
            acc[BACS_ACC_INVALID] += 1.f;
          }
          ypk[(i + h) >> 2] |= y8 << (8 * ((i + h) & 3));
        }
      }
    }

    // ---- seen heads: sigmoid(max_t up-sample(z_t)) and the focal head's logit, heads outer / pixels inner ------------
    // (x16 align_corners=True: the thread's SX pixels touch the low-res columns cb, cb+1, cb+2 only)
    float Lseen[SX], Lzf[SX], Lwx1[SX];
    uint32_t fdm = 0;  // bit i: pixel i's left tap is column cb+1 (else cb); its right tap is the next column, clamped
    const int cb = (!PSEUDO && EXACT && a.z) ? lerp_align_corners(SX * j, a.w, p.sx).i0 : 0;
    if (!PSEUDO && EXACT && a.z) {  // (the plan accepts the seen logits at the exact geometry only)
      float wx1[SX], zmx[SX], zf[SX];
#pragma unroll
      for (int i = 0; i < SX; ++i) {
        const Lerp lx = lerp_align_corners(SX * j + i, a.w, p.sx);
        wx1[i] = lx.w1;
        fdm |= (uint32_t)(lx.i0 - cb) << i;
        zmx[i] = -INFINITY;
        zf[i] = 0.f;
      }
      const float* zrow = zr + (size_t)r * a.T * a.w;
      const int c1 = min(cb + 1, a.w - 1), c2 = min(cb + 2, a.w - 1);
#pragma unroll 1
      for (int t = 0; t < a.T; ++t) {
        const float z0 = zrow[t * a.w + cb], z1 = zrow[t * a.w + c1], z2 = zrow[t * a.w + c2];
        const bool foc = t == a.focal_head;
#pragma unroll
        for (int i = 0; i < SX; ++i) {
          const bool up = (fdm >> i) & 1u;  // (c1, c2 are clamped like ATen's i1, so the right tap needs no case)
          const float za = up ? z1 : z0;
          const float zb = up ? z2 : z1;
          const float v = __fadd_rn(__fmul_rn(1.f - wx1[i], za), __fmul_rn(wx1[i], zb));
          zmx[i] = fmaxf(zmx[i], v);
          if (foc) zf[i] = v;
        }
      }
#pragma unroll
      for (int i = 0; i < SX; ++i) {
        Lseen[i] = sigmoid_fast(zmx[i]);
        Lzf[i] = zf[i];
        Lwx1[i] = wx1[i];
      }
    }

    // ---- pass 1a: max / arg-max (ties -> lowest channel) ------------------------------------------------------------
    float mx[SX];
    {
      int am[SX];
#pragma unroll
      for (int i = 0; i < SX; ++i) {
        mx[i] = -INFINITY;
        am[i] = 0;
      }
#pragma unroll 1
      for (int c = 0; c < K; ++c) {
        float vj, dl, dr;
        trio(c, vj, dl, dr);
#pragma unroll
        for (int i = 0; i < SX; ++i) {
          const float x = fmaf(BACS_LR_S(i), BACS_LR_LEFT(i) ? dl : dr, vj);
          if (x > mx[i]) {
            mx[i] = x;
            am[i] = c;
          }
        }
      }
      if constexpr (PSEUDO) {  // the arg-max replaces the label where it is 0; nothing else is written
#pragma unroll
        for (int i = 0; i < SX; ++i)
          if ((bg >> i) & 1u) a.preds[pix0 + i] = am[i];
        return;
      }
      if (a.preds) {
        int64_t* out = a.preds + pix0;
        if (EXACT && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
#pragma unroll
          for (int i = 0; i < SX; i += 2)
            *reinterpret_cast<longlong2*>(out + i) = make_longlong2((long long)am[i], (long long)am[i + 1]);
        } else {
#pragma unroll
          for (int i = 0; i < SX; ++i)
            if (EXACT || i < npx) out[i] = am[i];
        }
      }
    }

    // ---- pass 1b: exponent sums; channel 0 stays out (S_fg is accumulated directly) -----------------------------
    F2 so2[SX / 2], sn2[SX / 2];
#pragma unroll
    for (int ip = 0; ip < SX / 2; ++ip) {
      nm2[ip] = f2(-mx[2 * ip] * kLog2e, -mx[2 * ip + 1] * kLog2e);
      so2[ip] = sn2[ip] = f2b(0.f);
    }
    const F2 l2e2 = f2b(kLog2e);
    // exp2((v_j + s_i D) log2e - max log2e) of one pixel pair
    // (the two up-sampled logits come from scalar FFMAs with immediate s_i -- a packed FFMA2 would need the constant
    // pair in registers, re-materialised per channel -- and are identical to the values of pass 1a)
    auto exp_pair = [&](int ip, float s_lo, float s_hi, float side_lo, float side_hi, float vj) {
      const F2 arg = fma2(f2(fmaf(s_lo, side_lo, vj), fmaf(s_hi, side_hi, vj)), l2e2, nm2[ip]);
      return f2(ex2_fast(f2lo(arg)), ex2_fast(f2hi(arg)));
    };
#pragma unroll 1
    for (int c = 1; c < old_cl; ++c) {
      float vj, dl, dr;
      trio(c, vj, dl, dr);
#pragma unroll
      for (int ip = 0; ip < SX / 2; ++ip)
        so2[ip] = add2(so2[ip], exp_pair(ip, BACS_LR_S(2 * ip), BACS_LR_S(2 * ip + 1), BACS_LR_LEFT(2 * ip) ? dl : dr,
                                       BACS_LR_LEFT(2 * ip + 1) ? dl : dr, vj));
    }
#pragma unroll 1
    for (int c = max(old_cl, 1); c < K; ++c) {
      float vj, dl, dr;
      trio(c, vj, dl, dr);
#pragma unroll
      for (int ip = 0; ip < SX / 2; ++ip)
        sn2[ip] = add2(sn2[ip], exp_pair(ip, BACS_LR_S(2 * ip), BACS_LR_S(2 * ip + 1), BACS_LR_LEFT(2 * ip) ? dl : dr,
                                       BACS_LR_LEFT(2 * ip + 1) ? dl : dr, vj));
    }

    // ---- per-pixel terms: a rolled loop over dynamically indexed copies (local memory, L1) --------------------------
    float Lmx[SX], Lso[SX], Lsn[SX], Lcg1[SX], Lcg2[SX], Lsx[SX];
    uint32_t Ly[SX / 4];
#pragma unroll
    for (int i = 0; i < SX; ++i) {
      Lmx[i] = mx[i];
      Lso[i] = (i & 1) ? f2hi(so2[i >> 1]) : f2lo(so2[i >> 1]);
      Lsn[i] = (i & 1) ? f2hi(sn2[i >> 1]) : f2lo(sn2[i >> 1]);
      if constexpr (!EXACT) {
        Lsx[i] = sxr[i];
        Lcg1[i] = Lcg2[i] = 0.f;  // pixels past the span: no gradient in pass 2
      }
    }
#pragma unroll
    for (int q = 0; q < SX / 4; ++q) Ly[q] = ypk[q];
    float v0, dl0, dr0;
    trio(0, v0, dl0, dr0);
    float fa0 = 0.f, fa1 = 0.f, fa2 = 0.f;                              // focal gradient at columns cb, cb+1, cb+2
    uint32_t mbits = 0;
#pragma unroll 1
    for (int i = 0; i < (EXACT ? SX : npx); ++i) {
      const float sI = EXACT ? ((float)i + 0.5f) * kInvSX - 0.5f : Lsx[i];
      const bool left = EXACT ? i < SX / 2 : sI < 0.f;
      const uint32_t y8 = (Ly[i >> 2] >> (8 * (i & 3))) & 255u;
      const bool is_ign = y8 == 255u;
      const int y = is_ign ? -1 : (int)y8;
      const float mxi = Lmx[i];
      const float nmi = -mxi * kLog2e;
      const float x0 = fmaf(sI, left ? dl0 : dr0, v0);
      const float e0 = ex2_fast(fmaf(x0, kLog2e, nmi));
      const float S_fg = Lso[i] + Lsn[i];
      const float S = S_fg + e0;
      const float S_old = Lso[i] + (old_cl >= 1 ? e0 : 0.f);
      float xy = x0;
      if (y > 0) {
        float vj, dl, dr;
        trio(y, vj, dl, dr);
        xy = fmaf(sI, left ? dl : dr, vj);
      }
      float seen = 0.f, zfoc = 0.f, wx1 = 0.f;
      int fd = 0, fhi = 0;
      if (EXACT && a.z) {
        seen = Lseen[i];
        zfoc = Lzf[i];
        wx1 = Lwx1[i];
        fd = (int)((fdm >> i) & 1u);
        fhi = min(cb + fd + 1, a.w - 1) - cb;
      }
      if (a.seen_max) seen = __ldg(a.seen_max + pix0 + i);
      PixCoef pc;
      float gfoc;
      uint8_t dm;
      pixel_terms(a, p.inv_n, s_norm, old_cl, y, is_ign, mxi, S, S_old, S_fg, e0, x0, xy, seen, have_seen, zfoc, acc,
                  pc, gfoc, dm);
      mbits |= (uint32_t)dm << i;
      Lcg1[i] = pc.cg1;
      Lcg2[i] = pc.cg2;
      const float g0 = fmaf(e0, pc.cg0, -pc.d0);
      G0 += g0;
      if (left) GL0 = fmaf(sI, g0, GL0);
      else GR0 = fmaf(sI, g0, GR0);
      if (EXACT && a.gz && gfoc != 0.f) {
        const float c_lo = gfoc * (1.f - wx1), c_hi = gfoc * wx1;
        fa0 += (fd == 0 ? c_lo : 0.f) + (fhi == 0 ? c_hi : 0.f);
        fa1 += (fd == 1 ? c_lo : 0.f) + (fhi == 1 ? c_hi : 0.f);
        fa2 += (fhi == 2 ? c_hi : 0.f);
      }
    }
#pragma unroll
    for (int ip = 0; ip < SX / 2; ++ip) {
      cg1p[ip] = f2(Lcg1[2 * ip], Lcg1[2 * ip + 1]);
      cg2p[ip] = f2(Lcg2[2 * ip], Lcg2[2 * ip + 1]);
    }
    if (EXACT && a.gz) {
      float* grow = gacc + (size_t)r * (a.w + 1) + cb;
      if (fa0 != 0.f) atomicAdd(grow, fa0);
      if (fa1 != 0.f) atomicAdd(grow + 1, fa1);
      if (fa2 != 0.f) atomicAdd(grow + 2, fa2);
    }
    if (a.distill_mask) {
      uint8_t* out = a.distill_mask + pix0;
      uint32_t mpk[SX / 4];
#pragma unroll
      for (int q = 0; q < SX / 4; ++q) {
        const uint32_t nib = (mbits >> (4 * q)) & 15u;
        mpk[q] = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
      }
      if (EXACT && (reinterpret_cast<uintptr_t>(out) & (SX - 1)) == 0) {
        if (SX == 16) *reinterpret_cast<uint4*>(out) = make_uint4(mpk[0], mpk[1], mpk[2 % (SX / 4)], mpk[3 % (SX / 4)]);
        else *reinterpret_cast<uint2*>(out) = make_uint2(mpk[0], mpk[1]);
      } else {
#pragma unroll
        for (int i = 0; i < SX; ++i)
          if (EXACT || i < npx) out[i] = (uint8_t)((mbits >> i) & 1u);
      }
    }
  }
  if constexpr (PSEUDO) return;

  // ---- pass 2: gradients, reduced over the thread's pixels in registers, over the CTA's rows in shared memory --------
  if (p.g32) {
    float* gimg = p.g32 + (int64_t)b * K * lh * lw;
    for (int c0 = 0; c0 < K; c0 += CH) {
      const int cn = min(CH, K - c0);
      if (active) {
#pragma unroll 1
        for (int c = c0; c < c0 + cn; ++c) {
          float G = G0, GL = GL0, GR = GR0;
          if (c > 0) {
            float vj, dl, dr;
            trio(c, vj, dl, dr);
            const F2 l2e2 = f2b(kLog2e);
            const bool is_old = c < old_cl;
            F2 G2 = f2b(0.f);
            float GLa = 0.f, GLb = 0.f, GRa = 0.f, GRb = 0.f;
#pragma unroll
            for (int ip = 0; ip < SX / 2; ++ip) {
              const bool lo_left = BACS_LR_LEFT(2 * ip), hi_left = BACS_LR_LEFT(2 * ip + 1);
              const F2 arg = fma2(f2(fmaf(BACS_LR_S(2 * ip), lo_left ? dl : dr, vj),
                                     fmaf(BACS_LR_S(2 * ip + 1), hi_left ? dl : dr, vj)), l2e2, nm2[ip]);
              const F2 e2 = f2(ex2_fast(f2lo(arg)), ex2_fast(f2hi(arg)));
              const F2 g2 = mul2(e2, is_old ? cg1p[ip] : cg2p[ip]);
              G2 = add2(G2, g2);
              if (lo_left) GLa = fmaf(BACS_LR_S(2 * ip), f2lo(g2), GLa);
              else GRa = fmaf(BACS_LR_S(2 * ip), f2lo(g2), GRa);
              if (hi_left) GLb = fmaf(BACS_LR_S(2 * ip + 1), f2hi(g2), GLb);
              else GRb = fmaf(BACS_LR_S(2 * ip + 1), f2hi(g2), GRb);
            }
            G = f2lo(G2) + f2hi(G2);
            GL = GLa + GLb;
            GR = GRa + GRb;
          }
          // -dy at the label's own channel (rare: only channels that occur among the thread's labels)
          if (c >= ymin && c <= ymax) {
            const float dy = label_dy(a, p.inv_n, s_norm, old_cl, c);
            if (dy != 0.f) {
#pragma unroll
              for (int i = 0; i < SX; ++i) {
                if (((ypk[i >> 2] >> (8 * (i & 3))) & 255u) == (uint32_t)c) {
                  G -= dy;
                  if (BACS_LR_LEFT(i)) GL = fmaf(BACS_LR_S(i), -dy, GL);
                  else GR = fmaf(BACS_LR_S(i), -dy, GR);
                }
              }
            }
          }
          // adjoint of trio(): columns j-1 / j / j+1 (border columns fold into j)
          float dvj = G + GL - GR, dvl = -GL, dvr = GR;
          if (j == 0) {
            dvj += dvl;
            dvl = 0.f;
          }
          if (j == lw - 1) {
            dvj += dvr;
            dvr = 0.f;
          }
          float* q = planes + ((size_t)r * CH + (c - c0)) * lw + j;
          q[0] = dvj;
          q[plane_sz] = dvl;
          q[2 * plane_sz] = dvr;
        }
      }
      __syncthreads();
      // rows -> source rows with their y-weights; one global fp32 RED per low-res cell of the chunk
      // (a warp takes a channel, a lane a column: every row's value is read once and feeds all source rows)
      for (int cc = wid; cc < cn; cc += kLowresThreads / 32) {
        for (int x = lane; x < lw; x += 32) {
          float* gout = gimg + ((int64_t)(c0 + cc) * lh + base) * lw + x;
          if (nsrc <= 2) {  // the usual case: a row group lies between two source rows
            float sum0 = 0.f, sum1 = 0.f;
            for (int rr = 0; rr < rows; ++rr) {
              const float* q = planes + ((size_t)rr * CH + cc) * lw + x;
              float v = q[0];
              if (x + 1 < lw) v += q[plane_sz + 1];
              if (x >= 1) v += q[2 * plane_sz - 1];
              sum0 = fmaf(wrow[rr], v, sum0);
              sum1 = fmaf(wrow[R + rr], v, sum1);
            }
            if (sum0 != 0.f) atomicAdd(gout, sum0);
            if (nsrc == 2 && sum1 != 0.f) atomicAdd(gout + lw, sum1);
          } else {
            float sum[kLowresMaxSrc];
#pragma unroll
            for (int n = 0; n < kLowresMaxSrc; ++n) sum[n] = 0.f;
            for (int rr = 0; rr < rows; ++rr) {
              const float* q = planes + ((size_t)rr * CH + cc) * lw + x;
              float v = q[0];
              if (x + 1 < lw) v += q[plane_sz + 1];
              if (x >= 1) v += q[2 * plane_sz - 1];
#pragma unroll
              for (int n = 0; n < kLowresMaxSrc; ++n)
                if (n < nsrc) sum[n] = fmaf(wrow[n * R + rr], v, sum[n]);
            }
#pragma unroll
            for (int n = 0; n < kLowresMaxSrc; ++n)
              if (n < nsrc && sum[n] != 0.f) atomicAdd(gout + (int64_t)n * lw, sum[n]);
          }
        }
      }
      __syncthreads();
    }
  }
#undef BACS_LR_S
#undef BACS_LR_LEFT
  __syncthreads();

  if (a.gz) {
    float* g = a.gz + (int64_t)b * a.h * a.w;
    for (int idx = tid; idx < rows * a.w; idx += kLowresThreads) {
      const int rr = idx / a.w, i = idx - rr * a.w;
      const float v = gacc[rr * (a.w + 1) + i];
      if (v != 0.f) {
        const Lerp ly = lerp_align_corners(y0 + rr, a.h, p.sy);
        atomicAdd(g + ly.i0 * a.w + i, (1.f - ly.w1) * v);
        if (ly.w1 != 0.f) atomicAdd(g + ly.i1 * a.w + i, ly.w1 * v);
      }
    }
  }

  // ---- per-CTA partial sums ------------------------------------------------------------------------------------------
#pragma unroll
  for (int i = 0; i < BACS_NACC; ++i) {
    const float v = warp_sum(acc[i]);
    if (lane == 0) red_scratch[wid][i] = v;
  }
  __syncthreads();
  if (tid < BACS_NACC) {
    double v = 0.0;
    for (int wv = 0; wv < kLowresThreads / 32; ++wv) v += (double)red_scratch[wv][tid];
    p.partials[(int64_t)blockIdx.x * BACS_NACC + tid] = v;
  }
}

// fp32 accumulator -> storage type of the logits
template <typename T>
__global__ void __launch_bounds__(256) lowres_cast_kernel(const float* __restrict__ g, T* __restrict__ out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i < n) out[i] = DT<T>::from_f(g[i]);
}

}  // namespace bacs
