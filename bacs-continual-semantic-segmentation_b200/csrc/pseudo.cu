// Pseudo-labelled background (loss/bacs_loss.py:205-210):
//   pseudo = argmax_c teacher(img)[:, c];  mask[mask == 0] = pseudo[mask == 0]
// in place on the int64 labels, in one launch and without a host synchronisation (the torch form needs two
// nonzero() calls).  Ties go to the lowest channel and every label other than 0 keeps its bits.
//
// bacs_pseudo_label reads full-resolution teacher logits [B,K_t,H,W]: one HBM pass, K_t * s + 8 + 8 * f0 bytes per
// pixel (s bytes per logit, f0 the background fraction).  bacs_pseudo_label_lowres reads the teacher's low-res
// sem_logits and evaluates the bilinear up-sample inside the arg-max: the PSEUDO instantiation of pixel_lowres_kernel,
// so the labels equal the `preds` of bacs_pixel_loss_lowres at the same sem_logits.
#include "pixel_lowres.cuh"

namespace bacs {

constexpr int kPseudoPx = 8;  // consecutive pixels of one image per thread: one 16-byte row segment of 16-bit logits
constexpr int kPseudoThreads = 256;

// the thread's kPseudoPx logits of one channel row (16-byte loads when `vec`, else the first n scalars)
__device__ __forceinline__ void pseudo_row(const float* q, bool vec, int n, float (&v)[kPseudoPx]) {
  if (vec) {
    const float4 lo = __ldg(reinterpret_cast<const float4*>(q)), hi = __ldg(reinterpret_cast<const float4*>(q) + 1);
    v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w;
    v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
  } else {
#pragma unroll
    for (int i = 0; i < kPseudoPx; ++i) v[i] = i < n ? __ldg(q + i) : 0.f;
  }
}
template <typename T>
__device__ __forceinline__ void pseudo_row(const T* q, bool vec, int n, float (&v)[kPseudoPx]) {
  if (vec) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(q));
    const T* h = reinterpret_cast<const T*>(&u);
#pragma unroll
    for (int i = 0; i < kPseudoPx; ++i) v[i] = DT<T>::to_f(h[i]);
  } else {
#pragma unroll
    for (int i = 0; i < kPseudoPx; ++i) v[i] = i < n ? DT<T>::to_f(q[i]) : 0.f;
  }
}

// Thread t owns pixels [8 g, 8 g + 8) of image b (the last group of an image may be shorter).  A thread whose pixels
// carry no 0 label loads no logit.  vec_logits: teacher base 16-byte aligned and H*W*s a multiple of 16, so every full
// group's channel rows are 16-byte aligned; vec_labels: the same for the labels (H*W even).
template <typename T>
__global__ void __launch_bounds__(kPseudoThreads) pseudo_label_kernel(const T* __restrict__ teacher,
                                                                      int64_t* __restrict__ labels, int K, int64_t HW,
                                                                      int64_t groups_per_image, int64_t n_groups,
                                                                      int vec_logits, int vec_labels) {
  const int64_t t = (int64_t)blockIdx.x * kPseudoThreads + threadIdx.x;
  const int64_t b = t / groups_per_image;
  const int64_t p0 = (t - b * groups_per_image) * kPseudoPx;
  const int n = (int)min((int64_t)kPseudoPx, HW - p0);
  pdl_wait();
  if (t >= n_groups) return;
  int64_t* lab = labels + b * HW + p0;
  uint32_t bg = 0;  // bit i: pixel i is labelled 0
  if (vec_labels && n == kPseudoPx) {
#pragma unroll
    for (int i = 0; i < kPseudoPx; i += 2) {
      const longlong2 v = *reinterpret_cast<const longlong2*>(lab + i);
      bg |= ((uint32_t)(v.x == 0) << i) | ((uint32_t)(v.y == 0) << (i + 1));
    }
  } else {
#pragma unroll
    for (int i = 0; i < kPseudoPx; ++i)
      if (i < n) bg |= (uint32_t)(lab[i] == 0) << i;
  }
  if (bg == 0) return;
  const bool vec = vec_logits && n == kPseudoPx;
  const T* q = teacher + b * K * HW + p0;
  float mx[kPseudoPx];
  int am[kPseudoPx];
#pragma unroll
  for (int i = 0; i < kPseudoPx; ++i) {
    mx[i] = -INFINITY;
    am[i] = 0;
  }
#pragma unroll 4
  for (int c = 0; c < K; ++c, q += HW) {
    float v[kPseudoPx];
    pseudo_row(q, vec, n, v);
#pragma unroll
    for (int i = 0; i < kPseudoPx; ++i)
      if (v[i] > mx[i]) {
        mx[i] = v[i];
        am[i] = c;
      }
  }
#pragma unroll
  for (int i = 0; i < kPseudoPx; ++i)
    if ((bg >> i) & 1u) lab[i] = am[i];
}

}  // namespace bacs

using namespace bacs;

extern "C" {

int bacs_pseudo_label(const void* teacher, int32_t dtype, int32_t B, int32_t K_t, int32_t H, int32_t W,
                      int64_t* labels, bacs_stream_t stream) {
  BACS_REQUIRE(teacher && labels, "bacs_pseudo_label: teacher and labels are required");
  BACS_REQUIRE(B > 0 && K_t > 0 && H > 0 && W > 0, "bacs_pseudo_label: bad shape B=%d K_t=%d H=%d W=%d", B, K_t, H, W);
  BACS_REQUIRE(dtype >= 0 && dtype <= BACS_F16, "bacs_pseudo_label: unknown dtype %d", dtype);
  const int64_t HW = (int64_t)H * W;
  const int64_t gpi = (HW + kPseudoPx - 1) / kPseudoPx, n_groups = gpi * B;
  BACS_REQUIRE((n_groups + kPseudoThreads - 1) / kPseudoThreads <= 0x7fffffff, "bacs_pseudo_label: too many pixels");
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  const int vec_logits = al16(teacher) && (HW * (int64_t)dtype_size(dtype)) % 16 == 0;
  const int vec_labels = al16(labels) && HW % 2 == 0;
  const dim3 grid((unsigned)((n_groups + kPseudoThreads - 1) / kPseudoThreads));
  cudaStream_t s = (cudaStream_t)stream;
  int rc = BACS_OK;
  BACS_DISPATCH_DTYPE(dtype, TT, {
    rc = launch_pixel_kernel("bacs_pseudo_label", true, pseudo_label_kernel<TT>, grid, dim3(kPseudoThreads), 0, s,
                             reinterpret_cast<const TT*>(teacher), labels, (int)K_t, HW, gpi, n_groups, vec_logits,
                             vec_labels);
  });
  if (rc != BACS_OK) return rc;
  BACS_CHECK_LAUNCH("bacs_pseudo_label");
  return BACS_OK;
}

int bacs_pseudo_label_lowres(const void* sem_logits, int32_t dtype, int32_t B, int32_t K_t, int32_t lh, int32_t lw,
                             int32_t H, int32_t W, int64_t* labels, bacs_stream_t stream) {
  BACS_REQUIRE(sem_logits && labels, "bacs_pseudo_label_lowres: sem_logits and labels are required");
  BACS_REQUIRE(B > 0 && K_t > 0 && H > 0 && W > 0, "bacs_pseudo_label_lowres: bad shape B=%d K_t=%d H=%d W=%d", B, K_t,
               H, W);
  BACS_REQUIRE(dtype >= 0 && dtype <= BACS_F16, "bacs_pseudo_label_lowres: unknown dtype %d", dtype);
  // the loss kernel's arguments at this geometry, CE without seen logits; labels and preds are the same tensor
  bacs_pixel_args a = {};
  a.logits = sem_logits;
  a.labels = labels;
  a.preds = labels;
  a.B = B;
  a.K = K_t;
  a.H = H;
  a.W = W;
  a.dtype = dtype;
  a.mode = BACS_PIX_CE;
  a.ignore_index = -1;
  LowresPlan plan;
  if (!make_lowres_plan(a, lh, lw, &plan)) {
    set_error("bacs_pseudo_label_lowres: unsupported geometry (H=%d W=%d lh=%d lw=%d K_t=%d): as bacs_pixel_loss_lowres, "
              "W == s*lw with s = 8 or 16 and H a multiple of lh, or lh == ceil(H/s) and lw == ceil(W/s) for s = 8 or "
              "16; lw <= 256, K_t <= 255, staging within %zu bytes of shared memory",
              H, W, lh, lw, K_t, kLowresMaxSmem);
    return BACS_ERR_UNSUPPORTED;
  }
  LowresParams p = {};
  p.a = a;
  p.lh = lh;
  p.lw = lw;
  p.R = plan.R;
  p.groups_per_image = plan.groups;
  p.nsrc_max = plan.nsrc_max;
  p.hy = hp_scale(lh, H);
  p.hx = hp_scale(lw, W);
  auto kern = plan.exact ? (plan.SX == 16 ? pixel_lowres_kernel<16, true, true> : pixel_lowres_kernel<8, true, true>)
                         : (plan.SX == 16 ? pixel_lowres_kernel<16, false, true> : pixel_lowres_kernel<8, false, true>);
  const int rc = launch_pixel_kernel("bacs_pseudo_label_lowres", false, kern, dim3(plan.grid), dim3(kLowresThreads),
                                     plan.smem, (cudaStream_t)stream, p);
  if (rc != BACS_OK) return rc;
  BACS_CHECK_LAUNCH("bacs_pseudo_label_lowres");
  return BACS_OK;
}

}  // extern "C"
