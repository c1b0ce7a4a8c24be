// Seen / unseen detector heads at feature resolution.
//   reference: networks/bg_detector.py:17-40 (classification_head.get_distance / predict),
//              100-165 (get_seen_map_task, forward_seen_before, get_seen_probs)
// z[b,t,q] = bias_t + sum_c w[t,c] * |sigmoid(f[b,c,q]) - sigmoid(proto[t,c])|
// A weighted L1 distance per task head: HBM/ALU work, no GEMM form (SURVEY 7).
#include <algorithm>
#include <type_traits>

#include "common.cuh"

namespace bacs {

constexpr int kSeenWarps = 8;

// PX consecutive pixels of one channel row as one (up to 16-byte) register vector, converted at the point of use
template <int BYTES> struct RawVec;
template <> struct RawVec<2> { using type = uint16_t; };
template <> struct RawVec<4> { using type = uint32_t; };
template <> struct RawVec<8> { using type = uint2; };
template <> struct RawVec<16> { using type = uint4; };
template <typename T, int PX>
__device__ __forceinline__ void unpack_px(const typename RawVec<sizeof(T) * PX>::type& r, float* v) {
  const T* e = reinterpret_cast<const T*>(&r);
#pragma unroll
  for (int i = 0; i < PX; ++i) v[i] = DT<T>::to_f(e[i]);
}

template <typename T, int PX>
__device__ __forceinline__ void load_px(const T* p, float* v) {
  if constexpr (PX == 1) {
    v[0] = DT<T>::to_f(p[0]);
  } else if constexpr (sizeof(T) == 4) {
    if constexpr (PX == 4) {
      const float4 t = *reinterpret_cast<const float4*>(p);
      v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
      const float2 t = *reinterpret_cast<const float2*>(p);
      v[0] = t.x; v[1] = t.y;
    }
  } else {
    if constexpr (PX == 4) {
      const uint2 t = *reinterpret_cast<const uint2*>(p);
      const T* e = reinterpret_cast<const T*>(&t);
      v[0] = DT<T>::to_f(e[0]); v[1] = DT<T>::to_f(e[1]); v[2] = DT<T>::to_f(e[2]); v[3] = DT<T>::to_f(e[3]);
    } else {
      const uint32_t t = *reinterpret_cast<const uint32_t*>(p);
      const T* e = reinterpret_cast<const T*>(&t);
      v[0] = DT<T>::to_f(e[0]); v[1] = DT<T>::to_f(e[1]);
    }
  }
}

// The heads as separate device arrays (the modules' own parameters: no gather launch in front of the kernel).
struct HeadRows {
  const float* w[32];
  const float* b[32];
};
// The same for bacs_seen_logits_many: up to kMaxTasks heads (2 KB of kernel parameters).
struct HeadRowsMany {
  const float* w[kMaxTasks];
  const float* b[kMaxTasks];
};

// A CTA covers 32*PX consecutive pixels of one image (lane -> PX adjacent pixels, one vector load per channel
// row) and a slice of the channels; its 8 warps stride over the slice.  The CS CTAs of a thread-block cluster
// split the channels and the leader adds their partial sums through distributed shared memory, so the grid
// has enough CTAs to fill the machine while the summation order stays fixed.
// Per channel the T (weight, sigmoid(proto)) pairs sit in one shared-memory row read with broadcast 128-bit loads.
// MANY (bacs_seen_logits_many): blockIdx.z picks the chunk of TMAX heads h0 .. h0 + TMAX - 1 that the CTA evaluates;
// the chunks of a pixel tile read the same features, the later ones mostly from L2.
template <typename T, int TMAX, int PX, bool MANY = false>
__global__ void __launch_bounds__(32 * kSeenWarps, (TMAX * PX <= 32 ? 3 : (TMAX * PX <= 48 ? 2 : 1))) seen_logits_kernel(const T* __restrict__ feat, int D, int hw,
                                                                       const float* __restrict__ proto,
                                                                       const float* __restrict__ weight,
                                                                       const float* __restrict__ bias, int Tn,
                                                                       int chunk, int cs, float* __restrict__ z,
                                                                       const std::conditional_t<MANY, HeadRowsMany, HeadRows> rows,
                                                                       float* __restrict__ zero_out) {
  extern __shared__ __align__(16) float smem[];
  constexpr int PS = 32 * PX;            // pixels per CTA
  constexpr int stride = 2 * TMAX;       // floats per channel row: w[0..TMAX) | sigmoid(proto)[0..TMAX)
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int tid = threadIdx.x;
  const int rank = (int)blockIdx.x % cs, pb = (int)blockIdx.x / cs;
  const int b = blockIdx.y;
  const int h0 = MANY ? (int)blockIdx.z * TMAX : 0;   // first head of this CTA
  const int Th = MANY ? min(TMAX, Tn - h0) : Tn;      // heads of this CTA
  const int q0 = pb * PS + lane * PX;
  const int per = (D + cs - 1) / cs;
  const int c_begin = rank * per, c_end = min(D, c_begin + per);
  float acc[PX][TMAX];
#pragma unroll
  for (int i = 0; i < PX; ++i)
#pragma unroll
    for (int t = 0; t < TMAX; ++t) acc[i][t] = 0.f;
  pdl_wait();
  pdl_trigger();
  const T* base = feat + (int64_t)b * D * hw + q0;
  const bool live = q0 < hw;  // hw is a multiple of PX: a lane's pixels are all inside or all outside
  for (int c0 = c_begin; c0 < c_end; c0 += chunk) {
    const int cn = min(chunk, c_end - c0);
    __syncthreads();
    for (int i = tid; i < TMAX * cn; i += 32 * kSeenWarps) {
      const int t = i / cn, c = i - t * cn;
      smem[c * stride + t] = t < Th ? (weight ? weight[(h0 + t) * D + c0 + c] : rows.w[h0 + t][c0 + c]) : 0.f;
      smem[c * stride + TMAX + t] = t < Th ? sigmoid_fast(proto[(h0 + t) * D + c0 + c]) : 0.f;
    }
    __syncthreads();
    // warp wid handles channels wid, wid + 8, ... of the chunk; U channel rows in flight per lane
    constexpr int U = PX >= 4 ? 8 : 4;
    for (int c = wid; c < cn; c += U * kSeenWarps) {
      using Raw = typename RawVec<sizeof(T) * PX>::type;
      Raw x[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int cc = c + u * kSeenWarps;
        x[u] = Raw{};
        if (cc < cn && live) x[u] = *reinterpret_cast<const Raw*>(base + (int64_t)(c0 + cc) * hw);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int cc = c + u * kSeenWarps;
        if (cc < cn) {
          float sx[PX];
          unpack_px<T, PX>(x[u], sx);
#pragma unroll
          for (int i = 0; i < PX; ++i) sx[i] = sigmoid_mufu(sx[i]);
          const float4* row = reinterpret_cast<const float4*>(smem + cc * stride);
          float tab[2 * TMAX];
#pragma unroll
          for (int k = 0; k < (2 * TMAX) / 4; ++k) {
            const float4 v = row[k];
            tab[4 * k] = v.x; tab[4 * k + 1] = v.y; tab[4 * k + 2] = v.z; tab[4 * k + 3] = v.w;
          }
          // heads t >= Th have weight 0 in the table: no predicate in the inner loop
#pragma unroll
          for (int t = 0; t < TMAX; ++t) {
            if constexpr (PX % 2 == 0) {
#pragma unroll
              for (int i = 0; i < PX; i += 2) {
                const F2 d = sub2(f2(sx[i], sx[i + 1]), f2b(tab[TMAX + t]));  // one FADD2 for two pixels
                acc[i][t] = fmaf(tab[t], fabsf(f2lo(d)), acc[i][t]);
                acc[i + 1][t] = fmaf(tab[t], fabsf(f2hi(d)), acc[i + 1][t]);
              }
            } else {
#pragma unroll
              for (int i = 0; i < PX; ++i) acc[i][t] = fmaf(tab[t], fabsf(sx[i] - tab[TMAX + t]), acc[i][t]);
            }
          }
        }
      }
    }
  }
  // this CTA is done with its channel table; the leader's xfer region below can overlap its table, so the pushes
  // wait (barrier.cluster.wait before them) until every CTA of the cluster, the leader included, has arrived here
  if (cs > 1) asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  __syncthreads();
  // cross-warp reduction through shared memory: red[warp][t][pixel], then across the cluster
  float* red = smem;
#pragma unroll
  for (int t = 0; t < TMAX; ++t)
    if (t < Th) {
#pragma unroll
      for (int i = 0; i < PX; ++i) red[(wid * Th + t) * PS + lane * PX + i] = acc[i][t];
    }
  __syncthreads();
  float* xfer = smem + kSeenWarps * Th * PS;  // [cs][Th][PS] in the leader's shared memory
  const int n_out = Th * PS;
  if (cs > 1) {
    // non-leaders push their CTA sums into the leader's xfer[rank]
    uint32_t remote;
    const uint32_t local = (uint32_t)__cvta_generic_to_shared(xfer + (size_t)rank * n_out);
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(0));
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (rank != 0) {
      for (int e = tid; e < n_out; e += 32 * kSeenWarps) {
        float s = 0.f;
#pragma unroll
        for (int g = 0; g < kSeenWarps; ++g) s += red[g * n_out + e];
        asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(remote + 4u * (uint32_t)e), "f"(s) : "memory");
      }
    }
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (rank != 0) return;
  }
  for (int e = tid; e < n_out; e += 32 * kSeenWarps) {
    const int t = e / PS, px = e - t * PS;
    float s = weight ? bias[h0 + t] : rows.b[h0 + t][0];
#pragma unroll
    for (int g = 0; g < kSeenWarps; ++g) s += red[g * n_out + e];
    for (int r = 1; r < cs; ++r) s += xfer[(size_t)r * n_out + e];
    const int q = pb * PS + px;
    if (q < hw) {
      z[((int64_t)b * Tn + h0 + t) * hw + q] = s;
      if (zero_out && h0 + t == 0) zero_out[(int64_t)b * hw + q] = 0.f;   // accumulator of the following pixel kernel
    }
  }
}

__global__ void __launch_bounds__(256) seen_upsample_kernel(const float* __restrict__ z, int BT, int h, int w, int H,
                                                            int W, float sy, float sx, int apply_sigmoid,
                                                            float* __restrict__ out) {
  const int64_t total = (int64_t)BT * H * W;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int X = (int)(i % W);
    const int Y = (int)((i / W) % H);
    const int64_t bt = i / ((int64_t)W * H);
    const Lerp ly = lerp_align_corners(Y, h, sy), lx = lerp_align_corners(X, w, sx);
    const float* p = z + bt * h * w;
    const float v00 = p[ly.i0 * w + lx.i0], v01 = p[ly.i0 * w + lx.i1];
    const float v10 = p[ly.i1 * w + lx.i0], v11 = p[ly.i1 * w + lx.i1];
    const float wx0 = 1.f - lx.w1, wy0 = 1.f - ly.w1;
    // same operation order as ATen's upsample_bilinear2d
    const float top = __fadd_rn(__fmul_rn(wx0, v00), __fmul_rn(lx.w1, v01));
    const float bot = __fadd_rn(__fmul_rn(wx0, v10), __fmul_rn(lx.w1, v11));
    float v = __fadd_rn(__fmul_rn(wy0, top), __fmul_rn(ly.w1, bot));
    if (apply_sigmoid) v = sigmoid_acc(v);
    out[i] = v;
  }
}

// One block per channel: dW[c] = s * sum_{b,q} gz * |sig(f) - sig(p)|, optional dfeat.
template <typename T>
__global__ void __launch_bounds__(512) seen_head_backward_kernel(const T* __restrict__ feat, int B, int D, int hw,
                                                                 const float* __restrict__ proto_t,
                                                                 const float* __restrict__ weight_t,
                                                                 const float* __restrict__ gz,
                                                                 const float* __restrict__ scale_dev,
                                                                 float* __restrict__ dweight, float* __restrict__ dbias,
                                                                 T* __restrict__ dfeat) {
  __shared__ float scratch[32];
  const int c = blockIdx.x;
  const float scale = scale_dev ? *scale_dev : 1.f;
  if (c == D) {  // extra block: bias gradient
    float s = 0.f;
    for (int i = threadIdx.x; i < B * hw; i += blockDim.x) s += gz[i];
    s = block_sum(s, scratch);
    if (threadIdx.x == 0) dbias[0] = s * scale;
    return;
  }
  const float sp = sigmoid_fast(proto_t[c]);
  const float wc = weight_t[c];
  float acc = 0.f;
  // threads are split over images (ib) and pixels (iq) so that no index needs a division
  constexpr int U = 4;
  const int tq = min((int)blockDim.x, ((hw + U - 1) / U + 31) / 32 * 32);  // threads along the pixel axis
  const int nb_par = max(1, (int)blockDim.x / tq);                          // images processed side by side
  const int ib = threadIdx.x / tq, iq = threadIdx.x - ib * tq;
  if (ib < nb_par) {
    for (int b = ib; b < B; b += nb_par) {
      const T* row = feat + ((int64_t)b * D + c) * hw;
      const float* g = gz + (int64_t)b * hw;
      T* drow = dfeat ? dfeat + ((int64_t)b * D + c) * hw : nullptr;
      for (int q0 = iq; q0 < hw; q0 += tq * U) {
        float x[U], gq[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int q = q0 + u * tq;
          x[u] = q < hw ? DT<T>::to_f(row[q]) : 0.f;
          gq[u] = q < hw ? g[q] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int q = q0 + u * tq;
          if (q < hw) {
            const float sx = sigmoid_fast(x[u]);
            const float d = sx - sp;
            acc = fmaf(gq[u], fabsf(d), acc);
            if (drow) {
              const float sg = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);
              drow[q] = DT<T>::from_f(scale * gq[u] * wc * sg * sx * (1.f - sx));
            }
          }
        }
      }
    }
  }
  acc = block_sum(acc, scratch);
  if (threadIdx.x == 0) dweight[c] = acc * scale;
}

// Vectorised variant (hw a multiple of 8, 16-byte aligned rows): a thread handles 8 consecutive pixels per step
// (one 16-byte feature load, two 16-byte gz loads, one 16-byte gradient store), three steps in flight.
template <typename T>
__global__ void __launch_bounds__(256, 4) seen_head_backward_vec_kernel(const T* __restrict__ feat, int B, int D, int hw,
                                                                     const float* __restrict__ proto_t,
                                                                     const float* __restrict__ weight_t,
                                                                     const float* __restrict__ gz,
                                                                     const float* __restrict__ scale_dev,
                                                                     float* __restrict__ dweight,
                                                                     float* __restrict__ dbias, T* __restrict__ dfeat) {
  __shared__ float scratch[32];
  const int c = blockIdx.x;
  const float scale = scale_dev ? *scale_dev : 1.f;
  if (c == D) {  // extra block: bias gradient
    float s = 0.f;
    const float4* g4 = reinterpret_cast<const float4*>(gz);
    for (int i = threadIdx.x; i < (B * hw) / 4; i += blockDim.x) {
      const float4 v = g4[i];
      s += (v.x + v.y) + (v.z + v.w);
    }
    s = block_sum(s, scratch);
    if (threadIdx.x == 0) dbias[0] = s * scale;
    return;
  }
  const float sp = sigmoid_fast(proto_t[c]);
  const float coef = scale * weight_t[c];
  const int ipr = hw >> 3;           // 8-pixel items per row
  const int items = B * ipr;
  float acc = 0.f;
  constexpr int U = 2;
  constexpr int EB = 8 * sizeof(T);  // bytes per item
  using Raw = typename RawVec<(EB > 16 ? 16 : EB)>::type;
  for (int i0 = threadIdx.x; i0 < items; i0 += U * blockDim.x) {
    Raw x[U][EB / 16 > 0 ? EB / 16 : 1];
    float4 ga[U], gb[U];
    int64_t off[U];
    bool on[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u * blockDim.x;
      on[u] = i < items;
      const int b = on[u] ? i / ipr : 0;
      const int q = on[u] ? (i - b * ipr) * 8 : 0;
      off[u] = ((int64_t)b * D + c) * hw + q;
      const Raw* src = reinterpret_cast<const Raw*>(feat + off[u]);
#pragma unroll
      for (int k = 0; k < (EB / 16 > 0 ? EB / 16 : 1); ++k) x[u][k] = on[u] ? src[k] : Raw{};
      const float4* gp = reinterpret_cast<const float4*>(gz + (int64_t)b * hw + q);
      ga[u] = on[u] ? gp[0] : make_float4(0.f, 0.f, 0.f, 0.f);
      gb[u] = on[u] ? gp[1] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (!on[u]) continue;
      const T* e8 = reinterpret_cast<const T*>(&x[u][0]);
      const float g8[8] = {ga[u].x, ga[u].y, ga[u].z, ga[u].w, gb[u].x, gb[u].y, gb[u].z, gb[u].w};
      T o8[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float sx = sigmoid_mufu(DT<T>::to_f(e8[e]));
        const float d = sx - sp;
        acc = fmaf(g8[e], fabsf(d), acc);
        const float sg = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);
        o8[e] = DT<T>::from_f(g8[e] * coef * sg * sx * (1.f - sx));
      }
      if (dfeat) {
        Raw* dst = reinterpret_cast<Raw*>(dfeat + off[u]);
        const Raw* o = reinterpret_cast<const Raw*>(o8);
#pragma unroll
        for (int k = 0; k < (EB / 16 > 0 ? EB / 16 : 1); ++k) dst[k] = o[k];
      }
    }
  }
  acc = block_sum(acc, scratch);
  if (threadIdx.x == 0) dweight[c] = acc * scale;
}

// scale = weight * ready * [#bg > 0] / #kept ; focal = scale * sum(focal terms)
__global__ void focal_scale_kernel(const double* __restrict__ acc, const int32_t* __restrict__ ready, float weight,
                                   float* __restrict__ scale_out, double* __restrict__ out2) {
  const double kept = acc[BACS_ACC_KEPT];
  const bool on = (ready == nullptr || *ready != 0) && acc[BACS_ACC_BG] > 0.0 && kept > 0.0;
  const double s = on ? (double)weight / kept : 0.0;
  if (scale_out) *scale_out = (float)s;
  if (out2) {
    out2[0] = s;
    out2[1] = s * acc[BACS_ACC_FOCAL];
  }
}

__global__ void focal_scale_loss_kernel(const double* __restrict__ acc, const int32_t* __restrict__ ready, float weight,
                                        float main_coef, int main_over_wsum, float* __restrict__ scale_out,
                                        float* __restrict__ loss_out) {
  const double kept = acc[BACS_ACC_KEPT];
  const bool on = (ready == nullptr || *ready != 0) && acc[BACS_ACC_BG] > 0.0 && kept > 0.0;
  const double s = on ? (double)weight / kept : 0.0;
  if (scale_out) *scale_out = (float)s;
  if (loss_out) {
    double main = (double)main_coef * acc[BACS_ACC_LOSS];
    if (main_over_wsum) main /= acc[BACS_ACC_WSUM];
    *loss_out = (float)(main + s * acc[BACS_ACC_FOCAL]);
  }
}

}  // namespace bacs

using namespace bacs;

// MANY: bacs_seen_logits_many, chunks of 32 heads over the grid's z dimension (the T = 32 plan per chunk).
template <bool MANY>
static int seen_logits_impl(const void* features, int dtype, int B, int D, int h, int w, const float* proto,
                            const float* weight, const float* bias,
                            const std::conditional_t<MANY, HeadRowsMany, HeadRows>& rows, int T, float* z,
                            float* zero_out, bacs_stream_t stream) {
  const char* name = MANY ? "bacs_seen_logits_many" : "bacs_seen_logits";
  BACS_REQUIRE(B > 0 && B < 65536 && D > 0 && h > 0 && w > 0, "%s: bad shape", name);
  if (MANY) BACS_REQUIRE(T > 0 && T <= kMaxTasks, "%s: T=%d not in [1,%d]", name, T, kMaxTasks);
  else BACS_REQUIRE(T > 0 && T <= 32, "%s: T=%d not in [1,32]", name, T);
  const int hw = h * w;
  const int n_ch = (T + 31) / 32;          // chunks of 32 heads (MANY), else 1
  const int th = MANY ? std::min(T, 32) : T;  // heads per CTA
  const int tmax = MANY ? 32 : (T <= 2 ? 2 : (T <= 4 ? 4 : (T <= 6 ? 6 : (T <= 8 ? 8 : (T <= 12 ? 12 : (T <= 16 ? 16 : 32))))));
  int px = tmax <= 8 ? 4 : (tmax <= 16 ? 2 : 1);   // measured: 4 pixels x 12 heads (112 registers) is slower than 2 x 12
  const size_t es = dtype_size(dtype);
  if (hw % px != 0 || (reinterpret_cast<uintptr_t>(features) % (px * es)) != 0) px = 1;
  const int ps = 32 * px;
  const int n_pb = (hw + ps - 1) / ps;
  // cluster size: split the channels while the whole grid still fits the machine in one wave
  const int per_sm = tmax * px <= 32 ? 3 : (tmax * px <= 48 ? 2 : 1);  // resident CTAs (register budget, see the kernel)
  int cs = 1;
  while (cs < 8 && (int64_t)n_pb * B * n_ch * cs * 2 <= (int64_t)per_sm * sm_count() && D / (2 * cs) >= 2 * kSeenWarps)
    cs *= 2;
  const int stride = 2 * tmax;
  const int per = (D + cs - 1) / cs;
  int chunk = (32 * 1024 / 4) / stride;  // table of <= 32 KB
  chunk = std::max(kSeenWarps, chunk / kSeenWarps * kSeenWarps);
  if (chunk > per) chunk = (per + kSeenWarps - 1) / kSeenWarps * kSeenWarps;
  const size_t table = (size_t)chunk * stride * sizeof(float);
  const size_t red = (size_t)(kSeenWarps + cs) * th * ps * sizeof(float);
  const size_t smem = std::max(table, red);
  cudaStream_t s = (cudaStream_t)stream;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(n_pb * cs), (unsigned)B, (unsigned)n_ch);
  cfg.blockDim = dim3(32 * kSeenWarps);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
#define LAUNCH_Z(TT, TM, PXV)                                                                                     \
  do {                                                                                                            \
    auto kern = seen_logits_kernel<TT, TM, PXV, MANY>;                                                            \
    if (smem > 48 * 1024) {                                                                                       \
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);         \
      if (e != cudaSuccess) {                                                                                     \
        set_error("%s: shared memory opt-in failed: %s", name, cudaGetErrorString(e));                           \
        return BACS_ERR_CUDA;                                                                                     \
      }                                                                                                           \
    }                                                                                                             \
    cudaError_t le = cudaLaunchKernelEx(&cfg, kern, reinterpret_cast<const TT*>(features), D, hw, proto, weight,  \
                                        bias, T, chunk, cs, z, rows, zero_out);                                   \
    if (le != cudaSuccess) {                                                                                      \
      set_error("%s: launch failed: %s", name, cudaGetErrorString(le));                                          \
      return BACS_ERR_CUDA;                                                                                       \
    }                                                                                                             \
  } while (0)
#define LAUNCH_Z_PX(TT, TM, PXV)     \
  do {                               \
    if (px == 1) LAUNCH_Z(TT, TM, 1); \
    else LAUNCH_Z(TT, TM, PXV);      \
  } while (0)
  BACS_DISPATCH_DTYPE(dtype, TT, {
    if constexpr (MANY) LAUNCH_Z(TT, 32, 1);
    else if (tmax == 2) LAUNCH_Z_PX(TT, 2, 4);
    else if (tmax == 4) LAUNCH_Z_PX(TT, 4, 4);
    else if (tmax == 6) LAUNCH_Z_PX(TT, 6, 4);
    else if (tmax == 8) LAUNCH_Z_PX(TT, 8, 4);
    else if (tmax == 12) LAUNCH_Z_PX(TT, 12, 2);
    else if (tmax == 16) LAUNCH_Z_PX(TT, 16, 2);
    else LAUNCH_Z(TT, 32, 1);
  });
#undef LAUNCH_Z_PX
#undef LAUNCH_Z
  BACS_CHECK_LAUNCH(name);
  return BACS_OK;
}

extern "C" {

int bacs_seen_logits(const void* features, int dtype, int B, int D, int h, int w, const float* proto,
                     const float* weight, const float* bias, int T, float* z, bacs_stream_t stream) {
  BACS_REQUIRE(features && proto && weight && bias && z, "bacs_seen_logits: null pointer");
  HeadRows rows = {};
  return seen_logits_impl<false>(features, dtype, B, D, h, w, proto, weight, bias, rows, T, z, nullptr, stream);
}

int bacs_seen_logits_heads(const void* features, int dtype, int B, int D, int h, int w, const float* proto,
                           const float* const* weight_rows_host, const float* const* bias_host, int T, float* z,
                           float* zero_out, bacs_stream_t stream) {
  BACS_REQUIRE(features && proto && weight_rows_host && bias_host && z, "bacs_seen_logits_heads: null pointer");
  BACS_REQUIRE(T > 0 && T <= 32, "bacs_seen_logits_heads: T=%d not in [1,32]", T);
  HeadRows rows = {};
  for (int t = 0; t < T; ++t) {
    BACS_REQUIRE(weight_rows_host[t] && bias_host[t], "bacs_seen_logits_heads: null head %d", t);
    rows.w[t] = weight_rows_host[t];
    rows.b[t] = bias_host[t];
  }
  return seen_logits_impl<false>(features, dtype, B, D, h, w, proto, nullptr, nullptr, rows, T, z, zero_out, stream);
}

int bacs_seen_logits_many(const void* features, int dtype, int B, int D, int h, int w, const float* proto,
                          const float* weight, const float* bias, const float* const* weight_rows_host,
                          const float* const* bias_host, int T, float* z, float* zero_out, bacs_stream_t stream) {
  BACS_REQUIRE(features && proto && z, "bacs_seen_logits_many: null pointer");
  BACS_REQUIRE(T > 0 && T <= kMaxTasks, "bacs_seen_logits_many: T=%d not in [1,%d]", T, kMaxTasks);
  HeadRowsMany rows = {};
  if (weight_rows_host) {   // the heads' own parameters
    BACS_REQUIRE(bias_host, "bacs_seen_logits_many: null pointer");
    for (int t = 0; t < T; ++t) {
      BACS_REQUIRE(weight_rows_host[t] && bias_host[t], "bacs_seen_logits_many: null head %d", t);
      rows.w[t] = weight_rows_host[t];
      rows.b[t] = bias_host[t];
    }
    weight = bias = nullptr;
  } else {                  // stacked weight [T,D] and bias [T]
    BACS_REQUIRE(weight && bias, "bacs_seen_logits_many: null pointer");
  }
  return seen_logits_impl<true>(features, dtype, B, D, h, w, proto, weight, bias, rows, T, z, zero_out, stream);
}

int bacs_seen_upsample(const float* z, int B, int T, int h, int w, int scale, int apply_sigmoid, float* out,
                       bacs_stream_t stream) {
  BACS_REQUIRE(z && out, "bacs_seen_upsample: null pointer");
  BACS_REQUIRE(B > 0 && T > 0 && h > 0 && w > 0 && scale > 0, "bacs_seen_upsample: bad shape");
  const int H = h * scale, W = w * scale;
  const int64_t total = (int64_t)B * T * H * W;
  int64_t blocks = (total + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  seen_upsample_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(z, B * T, h, w, H, W, ac_scale(h, H),
                                                                           ac_scale(w, W), apply_sigmoid, out);
  BACS_CHECK_LAUNCH("bacs_seen_upsample");
  return BACS_OK;
}

int bacs_seen_head_backward(const void* features, int dtype, int B, int D, int h, int w, const float* proto_t,
                            const float* weight_t, const float* gz, const float* scale_dev, float* dweight,
                            float* dbias, void* dfeatures, bacs_stream_t stream) {
  BACS_REQUIRE(features && proto_t && weight_t && gz && dweight && dbias, "bacs_seen_head_backward: null pointer");
  BACS_REQUIRE(B > 0 && D > 0 && h > 0 && w > 0, "bacs_seen_head_backward: bad shape");
  const int hw = h * w;
  cudaStream_t s = (cudaStream_t)stream;
  const bool vec = hw % 8 == 0 && (reinterpret_cast<uintptr_t>(features) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(gz) & 15) == 0 &&
                   (!dfeatures || (reinterpret_cast<uintptr_t>(dfeatures) & 15) == 0);
  BACS_DISPATCH_DTYPE(dtype, TT, {
    if (vec)
      seen_head_backward_vec_kernel<TT><<<D + 1, 256, 0, s>>>(reinterpret_cast<const TT*>(features), B, D, hw, proto_t,
                                                              weight_t, gz, scale_dev, dweight, dbias,
                                                              reinterpret_cast<TT*>(dfeatures));
    else
      seen_head_backward_kernel<TT><<<D + 1, 512, 0, s>>>(reinterpret_cast<const TT*>(features), B, D, hw, proto_t,
                                                          weight_t, gz, scale_dev, dweight, dbias,
                                                          reinterpret_cast<TT*>(dfeatures));
  });
  BACS_CHECK_LAUNCH("bacs_seen_head_backward");
  return BACS_OK;
}

int bacs_focal_scale(const double* acc, const int32_t* ready, float weight, float* scale_out, double* out2,
                     bacs_stream_t stream) {
  BACS_REQUIRE(acc, "bacs_focal_scale: null pointer");
  focal_scale_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(acc, ready, weight, scale_out, out2);
  BACS_CHECK_LAUNCH("bacs_focal_scale");
  return BACS_OK;
}

int bacs_focal_scale_loss(const double* acc, const int32_t* ready, float weight, float main_coef, int main_over_wsum,
                          float* scale_out, float* loss_out, bacs_stream_t stream) {
  BACS_REQUIRE(acc, "bacs_focal_scale_loss: null pointer");
  focal_scale_loss_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(acc, ready, weight, main_coef, main_over_wsum, scale_out,
                                                             loss_out);
  BACS_CHECK_LAUNCH("bacs_focal_scale_loss");
  return BACS_OK;
}

}  // extern "C"
