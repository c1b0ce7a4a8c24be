// Prototype kernels: label-masked segmented reduction of penultimate features into
// per-task sums (reference-exact row split or per-channel), running-mean update.
//   reference: loss/prototypes.py:127-163 (update_feats_prototypes), 31-40 (ready)
#include "common.cuh"

namespace bacs {

// Per (image b, channel c) the masked pixels of task g form one run of n_bg elements in
// the reference's flattened masked-index tensor, at flat position
//     base = D * sum_{b'<b} n_b'g + c * n_bg .
// `.view(D, -1)` cuts that sequence into D rows of N_g elements, so the run spans at most
// two rows: r0 = base / N_g gets the elements with rank < split, r0 + 1 the rest, where
// split = (r0 + 1) * N_g - base.  Per-channel mode is the same code with split = n_bg.
// Each lane accumulates into its own column of a warp-private shared-memory table
// acc[task][low/high][lane] (conflict-free, no atomics): a pixel touches exactly one entry, so
// the cost per element does not grow with the number of tasks.
// VIEW (global view of a data-parallel batch, exact mode): pre and N_g also count the masked pixels of the images of
// other ranks -- view_pre[g] (images of lower ranks, added to pre) and view_n[g] (all ranks, in place of N_g) -- so the
// rows are those of one process fed every rank's images in rank order.  view_n[g] < 0 marks a view that could not be
// formed (peer time-out): such a task adds nothing and its count comes out as -inf, which makes every later running-mean
// update skip it.
// MANY (more than kTaskWindow tasks): blockIdx.z picks a window of kTaskWindow tasks; the block sums only the pixels of
// those tasks and writes their columns, so its shared memory and split bookkeeping are those of a 32-task launch.
constexpr int kAccWarps = 8;
constexpr int kTaskWindow = 32;
template <typename T, bool MANY = false, bool VIEW = false>
__global__ void __launch_bounds__(32 * kAccWarps) proto_accumulate_kernel(const T* __restrict__ feat, int B, int D,
                                                                          int hw, const int8_t* __restrict__ task,
                                                                          const int32_t* __restrict__ rank,
                                                                          const int32_t* __restrict__ n_bt, int Tn,
                                                                          int mode,
                                                                          float* __restrict__ partial /* [B,D,Tn,2] */,
                                                                          const void* __restrict__ count_raw, int count_is_int64,
                                                                          unsigned long long* __restrict__ count_snap,
                                                                          const long long* __restrict__ view_pre,
                                                                          const long long* __restrict__ view_n) {
  extern __shared__ float s_acc[];  // [warp][Tw][2][32]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const int c = blockIdx.x * kAccWarps + wid;
  const int t_lo = MANY ? (int)blockIdx.z * kTaskWindow : 0;      // first task of this block
  const int Tw = MANY ? min(kTaskWindow, Tn - t_lo) : Tn;         // tasks of this block
  pdl_wait();
  pdl_trigger();
  if (count_snap && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < Tw)
    count_snap[t_lo + threadIdx.x] = count_is_int64 ? reinterpret_cast<const unsigned long long*>(count_raw)[t_lo + threadIdx.x]
                                                    : (unsigned long long)reinterpret_cast<const unsigned*>(count_raw)[t_lo + threadIdx.x];
  if (c >= D) return;
  float* acc = s_acc + (size_t)wid * Tw * 64;
  for (int i = lane; i < Tw * 64; i += 32) acc[i] = 0.f;
  // lane g holds the split point of task t_lo + g
  int split = 0x7fffffff;
  if (mode == 0 && lane < Tw) {
    long long pre = 0, tot = 0;
    for (int bb = 0; bb < B; ++bb) {
      const int n = n_bt[bb * Tn + t_lo + lane];
      if (bb < b) pre += n;
      tot += n;
    }
    if constexpr (VIEW) {
      pre += view_pre[t_lo + lane];
      tot = view_n[t_lo + lane];
    }
    const long long nb = n_bt[b * Tn + t_lo + lane];
    if (tot > 0) {
      const long long base = (long long)D * pre + (long long)c * nb;
      const long long r0 = base / tot;
      const long long sp = (r0 + 1) * tot - base;
      split = sp > 0x7fffffffLL ? 0x7fffffff : (int)sp;
    }
  }
  __syncwarp();
  const T* row = feat + ((int64_t)b * D + c) * hw;
  const int8_t* tk = task + (int64_t)b * hw;
  const int32_t* rk = rank + (int64_t)b * hw;
  constexpr int U = 4;  // independent loads in flight per lane
  for (int q0 = 0; q0 < hw; q0 += 32 * U) {
    int t[U], k[U];
    float v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int q = q0 + u * 32 + lane;
      t[u] = q < hw ? (int)tk[q] : -1;
      if constexpr (MANY) t[u] = (t[u] >= t_lo && t[u] < t_lo + Tw) ? t[u] - t_lo : -1;
      v[u] = (t[u] >= 0) ? DT<T>::to_f(row[q]) : 0.f;
      k[u] = (t[u] >= 0) ? rk[q] : 0;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int sp = __shfl_sync(0xffffffffu, split, t[u] < 0 ? 0 : t[u]);
      if (t[u] >= 0) acc[(t[u] * 2 + (k[u] < sp ? 0 : 1)) * 32 + lane] += v[u];
    }
  }
  __syncwarp();
  float* out = partial + (((int64_t)b * D + c) * Tn + t_lo) * 2;
  for (int e = 0; e < Tw * 2; ++e) {
    const float r = warp_sum(acc[e * 32 + lane]);
    if (lane == 0) out[e] = r;
  }
}

// Vectorised variant (hw a multiple of 8, 16-byte aligned rows): a lane handles 8 consecutive pixels per step; task
// bytes and features of a row's first step are requested before the split points are worked out.  The per-warp table
// has one 32-float row per (task, low / high) entry: a lane only ever touches its own bank.
template <typename T, bool MANY = false, bool VIEW = false>
__global__ void __launch_bounds__(32 * kAccWarps, 4) proto_accumulate_vec_kernel(const T* __restrict__ feat, int B, int D,
                                                                                 int hw, const int8_t* __restrict__ task,
                                                                                 const int32_t* __restrict__ rank,
                                                                                 const int32_t* __restrict__ n_bt, int Tn,
                                                                                 int mode, float* __restrict__ partial,
                                                                                 const void* __restrict__ count_raw,
                                                                                 int count_is_int64,
                                                                                 unsigned long long* __restrict__ count_snap,
                                                                                 const long long* __restrict__ view_pre,
                                                                                 const long long* __restrict__ view_n) {
  extern __shared__ float s_acc[];  // [warp][Tw*2 + 2][32] | [warp][33] split points
  __shared__ long long s_pre[32], s_tot[32];  // per task: masked pixels in the images before b / in all images
  __shared__ int s_nb[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const int c = blockIdx.x * kAccWarps + wid;
  const int t_lo = MANY ? (int)blockIdx.z * kTaskWindow : 0;
  const int Tw = MANY ? min(kTaskWindow, Tn - t_lo) : Tn;
  const bool live = c < D;
  pdl_wait();
  pdl_trigger();
  // The row's first loads go out before anything else: task bytes, features and ranks of a step are all in flight
  // together while the split points are worked out.
  const T* row = feat + ((int64_t)b * D + (live ? c : 0)) * hw;
  const int8_t* tk = task + (int64_t)b * hw;
  const int32_t* rk = rank + (int64_t)b * hw;
  const int items = hw >> 3;
  constexpr int U = 4;
  constexpr int NV = sizeof(T) == 4 ? 2 : 1;  // 16-byte vectors per 8 pixels
  uint2 t8[U];
  uint4 raw[U][NV];
  int4 r0[U], r1[U];
  auto load_step = [&](int it0) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int it = it0 + u * 32 + lane;
      const bool ok = live && it < items;
      t8[u] = ok ? *reinterpret_cast<const uint2*>(tk + it * 8) : make_uint2(0xffffffffu, 0xffffffffu);
#pragma unroll
      for (int k = 0; k < NV; ++k) raw[u][k] = ok ? reinterpret_cast<const uint4*>(row + it * 8)[k] : make_uint4(0u, 0u, 0u, 0u);
    }
  };
  auto load_ranks = [&](int it0) {   // shared by the D channel rows of the image: L2 hits, fetched after the split points
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int it = it0 + u * 32 + lane;
      r0[u] = r1[u] = make_int4(0, 0, 0, 0);
      if (mode == 0 && it < items) {
        r0[u] = *reinterpret_cast<const int4*>(rk + it * 8);
        r1[u] = *reinterpret_cast<const int4*>(rk + it * 8 + 4);
      }
    }
  };
  load_step(0);
  // fused update: the finalize launch reads the counts of BEFORE the step from this snapshot while one of its blocks
  // already writes the new ones (8 bytes per task whatever the count type; a float count sits in the low word)
  if (count_snap && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < Tw)
    count_snap[t_lo + threadIdx.x] = count_is_int64 ? reinterpret_cast<const unsigned long long*>(count_raw)[t_lo + threadIdx.x]
                                                    : (unsigned long long)reinterpret_cast<const unsigned*>(count_raw)[t_lo + threadIdx.x];
  if (mode == 0) {  // the same for all channels of the block: warp w takes tasks w, w + 8, ..., its lanes the images
    for (int t = wid; t < Tw; t += kAccWarps) {
      long long pre = 0, tot = 0;
      for (int bb = lane; bb < B; bb += 32) {
        const int n = n_bt[bb * Tn + t_lo + t];
        if (bb < b) pre += n;
        tot += n;
      }
      pre = warp_sum(pre);
      tot = warp_sum(tot);
      if constexpr (VIEW) {
        pre += view_pre[t_lo + t];
        tot = view_n[t_lo + t];
      }
      if (lane == 0) {
        s_pre[t] = pre;
        s_tot[t] = tot;
        s_nb[t] = n_bt[b * Tn + t_lo + t];
      }
    }
  }
  __syncthreads();
  if (!live) return;
  const int ne = Tw * 2;
  float* acc = s_acc + (size_t)wid * (ne + 2) * 32;          // + the dump entry of pixels without a task
  int* s_split = reinterpret_cast<int*>(s_acc + (size_t)kAccWarps * (ne + 2) * 32) + wid * 33;
  for (int i = lane; i < (ne + 2) * 32; i += 32) acc[i] = 0.f;
  int split = 0x7fffffff;
  if (mode == 0 && lane < Tw) {
    const long long tot = s_tot[lane], nb = s_nb[lane];
    if (tot > 0) {
      const long long base = (long long)D * s_pre[lane] + (long long)c * nb;
      long long q0;
      if ((long long)D * tot < 0x7fffffffLL) q0 = (long long)((unsigned)base / (unsigned)tot);  // 32-bit division
      else q0 = base / tot;
      const long long sp = (q0 + 1) * tot - base;
      split = sp > 0x7fffffffLL ? 0x7fffffff : (int)sp;
    }
  }
  s_split[lane] = split;                    // lanes >= Tw hold INT_MAX: the dump entry (index Tw) never splits
  if (lane == 0) s_split[32] = 0x7fffffff;
  __syncwarp();
  // Branch-free inner loop: a pixel without a task (-1: background / ignore / later task) adds into a dump entry
  // (table row Tn, split point INT_MAX) instead of taking a branch.
  for (int it0 = 0; it0 < items; it0 += 32 * U) {
    if (it0 > 0) load_step(it0);
    load_ranks(it0);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (((~t8[u].x | ~t8[u].y) & 0x80808080u) == 0u) continue;   // no byte >= 0 in this lane's 8 pixels
      const int rr[8] = {r0[u].x, r0[u].y, r0[u].z, r0[u].w, r1[u].x, r1[u].y, r1[u].z, r1[u].w};
      const T* e8 = reinterpret_cast<const T*>(&raw[u][0]);
      // labels are blocky: 8 pixels of ONE task whose ranks (increasing along the row) lie on one side of the split
      // point are added in registers and cost a single table update
      unsigned t0 = t8[u].x & 0xffu;
      if (t8[u].x == t0 * 0x01010101u && t8[u].y == t8[u].x) {
        if constexpr (MANY) {   // 8 pixels of one task outside the window add nothing here
          t0 -= (unsigned)t_lo;
          if (t0 >= (unsigned)Tw) continue;
        }
        const int sp = s_split[t0];
        if (rr[7] < sp || rr[0] >= sp) {
          float v = 0.f;
#pragma unroll
          for (int e = 0; e < 8; ++e) v += DT<T>::to_f(e8[e]);
          acc[(int)t0 * 64 + (rr[0] < sp ? 0 : 32) + lane] += v;
          continue;
        }
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const unsigned tb = ((e < 4 ? t8[u].x >> (8 * e) : t8[u].y >> (8 * (e - 4))) & 0xffu);
        // 0xff (-1) -> the dump entry; so does a task outside the window (the subtraction wraps below it)
        const int tt = MANY ? (int)min(tb - (unsigned)t_lo, (unsigned)Tw) : (int)min(tb, (unsigned)Tn);
        const int hi = rr[e] < s_split[tt] ? 0 : 32;
        acc[tt * 64 + hi + lane] += DT<T>::to_f(e8[e]);         // bank = lane: conflict-free whatever the tasks
      }
    }
  }
  __syncwarp();
  // The ne column sums of the warp as a reduce-scatter over groups of 16 entries: after the exchange with lane ^ 16 a
  // lane keeps 8 entries, then 4, 2, 1 -- 16 shuffles per group instead of 5 per entry, and the same association
  // ((l, l^16), then ^8, ^4, ^2, ^1) as warp_sum(), so the sums are bit-identical to the entry-by-entry form.
  float* out = partial + (((int64_t)b * D + c) * Tn + t_lo) * 2;
  for (int e0 = 0; e0 < ne; e0 += 16) {
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = e0 + i < ne ? acc[(e0 + i) * 32 + lane] : 0.f;
    float k8[8], k4[4], k2[2];
    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2;
#pragma unroll
    for (int i = 0; i < 8; ++i) k8[i] = (b4 ? v[i + 8] : v[i]) + __shfl_xor_sync(0xffffffffu, b4 ? v[i] : v[i + 8], 16);
#pragma unroll
    for (int i = 0; i < 4; ++i) k4[i] = (b3 ? k8[i + 4] : k8[i]) + __shfl_xor_sync(0xffffffffu, b3 ? k8[i] : k8[i + 4], 8);
#pragma unroll
    for (int i = 0; i < 2; ++i) k2[i] = (b2 ? k4[i + 2] : k4[i]) + __shfl_xor_sync(0xffffffffu, b2 ? k4[i] : k4[i + 2], 4);
    float k1 = (b1 ? k2[1] : k2[0]) + __shfl_xor_sync(0xffffffffu, b1 ? k2[0] : k2[1], 2);
    k1 += __shfl_xor_sync(0xffffffffu, k1, 1);
    const int e = e0 + ((lane >> 1) & 15);
    if ((lane & 1) == 0 && e < ne) out[e] = k1;
  }
}

// ---- the same sums as a one-hot GEMM on the tensor cores (16-bit features, hw a multiple of 32) ------------------------
// total[c][t] = sum_p feat[c][p] * [task(p) == t] is a [16 channels x pixels] x [pixels x 8 tasks] product per warp:
// mma.sync.m16n8k16 with the features as the row-major A fragments straight from NCHW (a lane loads 8 consecutive
// pixels of rows g and g + 8 with two 16-byte loads; which pixel sits in which k slot is free as long as B agrees) and
// the one-hot B fragments made in registers from the lane's own 8 task bytes (byte compare + byte permute): no shared
// memory, no per-pixel table update -- about 50 instructions per 1024-pixel channel row instead of 964.  The products
// are exact (0/1 times a 16-bit value), the accumulation is fp32.  Exact mode: a (channel, task) run that crosses a row
// boundary of the reference's D x N_g view (split point inside the image's n_bt pixels: about D / B channels per task)
// is re-read by the whole warp with the rank test; all other entries are "everything below the split point".
constexpr int kMmaWarps = 2;
template <typename T> struct MmaOne;
template <> struct MmaOne<__nv_bfloat16> { static constexpr uint32_t pair = 0x3F803F80u; };
template <> struct MmaOne<__half> { static constexpr uint32_t pair = 0x3C003C00u; };
template <typename T>
__device__ __forceinline__ void mma_16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                          uint32_t b1) {
  if constexpr (DT<T>::id == BACS_BF16)
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
  else
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

template <typename T, int NT, bool MANY = false, bool VIEW = false>  // NT = ceil(Tn / 8) task tiles (4 with MANY: one 32-task window)
__global__ void __launch_bounds__(32 * kMmaWarps) proto_accumulate_mma_kernel(const T* __restrict__ feat, int B, int D, int hw,
                                                                              const int8_t* __restrict__ task,
                                                                              const int32_t* __restrict__ rank,
                                                                              const int32_t* __restrict__ n_bt, int Tn, int mode,
                                                                              double* __restrict__ sums /* [Tn][D], zeroed */,
                                                                              const void* __restrict__ count_raw,
                                                                              int count_is_int64,
                                                                              unsigned long long* __restrict__ count_snap,
                                                                              const long long* __restrict__ view_pre,
                                                                              const long long* __restrict__ view_n) {
  static_assert(sizeof(T) == 2, "16-bit tensor-core operands");
  __shared__ long long s_pre[32], s_tot[32];
  __shared__ int s_nb[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const int cb = (blockIdx.x * kMmaWarps + wid) * 16;  // first channel of this warp
  const int g = lane >> 2, tig = lane & 3;
  const int t_lo = MANY ? (int)blockIdx.z * kTaskWindow : 0;
  const int Tw = MANY ? min(kTaskWindow, Tn - t_lo) : Tn;
  pdl_wait();
  pdl_trigger();
  if (count_snap && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < Tw)
    count_snap[t_lo + threadIdx.x] = count_is_int64 ? reinterpret_cast<const unsigned long long*>(count_raw)[t_lo + threadIdx.x]
                                                    : (unsigned long long)reinterpret_cast<const unsigned*>(count_raw)[t_lo + threadIdx.x];
  // the first loads go out before the split bookkeeping
  const bool live = cb < D;
  const T* rowA = feat + ((int64_t)b * D + (live ? cb : 0) + g) * hw + tig * 8;
  const T* rowB = rowA + (int64_t)8 * hw;
  const int8_t* tk = task + (int64_t)b * hw + tig * 8;
  constexpr int U = 8;  // 32-pixel chunks in flight per lane
  uint4 ra[U], rb[U];
  uint2 tw[U];
  auto load_step = [&](int q0) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int q = q0 + u * 32;
      if (live && q < hw) {
        ra[u] = __ldg(reinterpret_cast<const uint4*>(rowA + q));
        rb[u] = __ldg(reinterpret_cast<const uint4*>(rowB + q));
        tw[u] = __ldg(reinterpret_cast<const uint2*>(tk + q));
      } else {
        ra[u] = rb[u] = make_uint4(0u, 0u, 0u, 0u);
        tw[u] = make_uint2(0xffffffffu, 0xffffffffu);
      }
    }
  };
  load_step(0);
  if (mode == 0) {  // per task: masked pixels in the images before b / in all images / in this image
    for (int t = wid; t < Tw; t += kMmaWarps) {
      long long pre = 0, tot = 0;
      for (int bb = lane; bb < B; bb += 32) {
        const int n = n_bt[bb * Tn + t_lo + t];
        if (bb < b) pre += n;
        tot += n;
      }
      pre = warp_sum(pre);
      tot = warp_sum(tot);
      if constexpr (VIEW) {
        pre += view_pre[t_lo + t];
        tot = view_n[t_lo + t];
      }
      if (lane == 0) {
        s_pre[t] = pre;
        s_tot[t] = tot;
        s_nb[t] = n_bt[b * Tn + t_lo + t];
      }
    }
  }
  __syncthreads();
  if (!live) return;
  float d[NT][4];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) d[nt][0] = d[nt][1] = d[nt][2] = d[nt][3] = 0.f;
  for (int q0 = 0; q0 < hw; q0 += 32 * U) {
    if (q0 > 0) load_step(q0);
#pragma unroll
    for (int u = 0; u < U; ++u) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        // words (x, y) / (z, w) of the two rows: pixels 4j .. 4j+3 of the lane; k slots 2 tig + {0,1} and 2 tig + 8 + {0,1}
        const uint32_t a0 = j ? ra[u].z : ra[u].x, a1 = j ? rb[u].z : rb[u].x;
        const uint32_t a2 = j ? ra[u].w : ra[u].y, a3 = j ? rb[u].w : rb[u].y;
        const uint32_t tb = j ? tw[u].y : tw[u].x;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
          const uint32_t m = __vcmpeq4(tb, (uint32_t)(t_lo + 8 * nt + g) * 0x01010101u);  // 0xff where the pixel's task is this lane's n
          mma_16816<T>(d[nt], a0, a1, a2, a3, __byte_perm(m, 0u, 0x1100) & MmaOne<T>::pair,
                       __byte_perm(m, 0u, 0x3322) & MmaOne<T>::pair);
        }
      }
    }
  }
  // D fragment: d[nt][0..1] = (row g, tasks 8 nt + 2 tig + {0,1}), d[nt][2..3] = (row g + 8, same tasks).
  // The totals go straight into the [Tn][D] fp64 sums (no per-image partial buffer, no gather pass): an entry of image
  // b, channel c, task t lands in row r0 = (D pre_bt + c n_bt) / N_t of the reference's D x N_t view (row c in
  // per-channel mode).  The addends are fp32 values, about B per row: their fp64 sum is exact whatever the order.
  // A run that crosses a row boundary (split point inside the image's n_bt pixels: about D / B channels per task) is
  // re-read by the whole warp with the rank test and contributes to rows r0 and r0 + 1.
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int t = 8 * nt + 2 * tig + (e & 1), c = cb + g + (e >> 1) * 8;
      int row = c, sp = 0x7fffffff;
      bool is_split = false;
      if (t < Tw && mode == 0) {
        const long long tot = s_tot[t], nb = s_nb[t];
        if (tot > 0 && nb > 0) {
          const long long base = (long long)D * s_pre[t] + (long long)c * nb;
          long long q;
          if ((long long)D * tot < 0x7fffffffLL) q = (long long)((unsigned)base / (unsigned)tot);  // 32-bit division
          else q = base / tot;
          const long long spl = (q + 1) * tot - base;
          row = (int)q;
          is_split = spl < nb;
          sp = is_split ? (int)spl : 0x7fffffff;
        }
      }
      if (t < Tw && !is_split && d[nt][e] != 0.f && (!VIEW || s_tot[t] > 0)) atomicAdd(sums + (int64_t)(t_lo + t) * D + row, (double)d[nt][e]);
      unsigned todo = __ballot_sync(0xffffffffu, is_split);
      while (todo) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        const int sc = __shfl_sync(0xffffffffu, c, src), st = t_lo + __shfl_sync(0xffffffffu, t, src);
        const int ssp = __shfl_sync(0xffffffffu, sp, src), srow = __shfl_sync(0xffffffffu, row, src);
        const T* rowp = feat + ((int64_t)b * D + sc) * hw;
        const int8_t* tkr = task + (int64_t)b * hw;
        const int32_t* rkr = rank + (int64_t)b * hw;
        float lo = 0.f, hi = 0.f;
        for (int it = lane; it < (hw >> 3); it += 32) {
          const uint4 raw = __ldg(reinterpret_cast<const uint4*>(rowp + it * 8));
          const uint2 t8 = __ldg(reinterpret_cast<const uint2*>(tkr + it * 8));
          const int4 r0 = __ldg(reinterpret_cast<const int4*>(rkr + it * 8)), r1 = __ldg(reinterpret_cast<const int4*>(rkr + it * 8 + 4));
          const int rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
          const T* e8 = reinterpret_cast<const T*>(&raw);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const unsigned tbyte = ((k < 4 ? t8.x >> (8 * k) : t8.y >> (8 * (k - 4))) & 0xffu);
            if ((int)tbyte == st) {
              const float v = DT<T>::to_f(e8[k]);
              if (rr[k] < ssp) lo += v;
              else hi += v;
            }
          }
        }
        lo = warp_sum(lo);
        hi = warp_sum(hi);
        if (lane == 0) {
          atomicAdd(sums + (int64_t)st * D + srow, (double)lo);
          atomicAdd(sums + (int64_t)st * D + srow + 1, (double)hi);
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) proto_zero_sums_kernel(double* __restrict__ sums, int n) {
  pdl_wait();
  pdl_trigger();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) sums[i] = 0.0;
}

// One block per task g; thread r gathers the partial runs that land in output row r.
// Image b's masked elements occupy flat positions [D*pre_b, D*(pre_b+n_b)), i.e. rows
// lo_b .. hi_b of the D x N_g view; row r only looks at images with lo_b <= r <= hi_b + 1.
constexpr int kFinMaxB = 1024;
constexpr int kFinRows = 32;   // output rows per block
constexpr int kFinLanes = 8;   // images are strided over this many threads per row
template <bool VIEW = false>   // VIEW: rows of the global view (gather only, no fused update)
__global__ void __launch_bounds__(kFinRows* kFinLanes) proto_finalize_kernel(const float* __restrict__ partial, int B,
                                                                            int D, const int32_t* __restrict__ n_bt,
                                                                            int Tn, int mode,
                                                                            double* __restrict__ sums,
                                                                            double* __restrict__ counts,
                                                                            float* __restrict__ proto, void* __restrict__ count,
                                                                            int count_is_int64,
                                                                            const unsigned long long* __restrict__ count_snap,
                                                                            int32_t* __restrict__ ready, int gather,
                                                                            const long long* __restrict__ view_pre,
                                                                            const long long* __restrict__ view_n) {
  __shared__ long long s_pre[kFinMaxB];
  __shared__ int s_nb[kFinMaxB], s_lo[kFinMaxB], s_hi[kFinMaxB];
  __shared__ long long s_tot;
  __shared__ double s_red[kFinLanes][kFinRows];
  const int g = blockIdx.x;
  const int tid = threadIdx.x;
  pdl_wait();
  pdl_trigger();
  for (int bb = tid; bb < B; bb += blockDim.x) s_nb[bb] = n_bt[bb * Tn + g];  // parallel loads, serial scan below
  __syncthreads();
  if (tid == 0) {
    long long run = 0;
    if constexpr (VIEW) run = view_pre[g];
    for (int bb = 0; bb < B; ++bb) {
      s_pre[bb] = run;
      run += s_nb[bb];
    }
    if constexpr (VIEW) {   // the counts stay local: the exchange of the sums adds them up
      s_tot = view_n[g];
      if (blockIdx.y == 0) counts[g] = view_n[g] < 0 ? -INFINITY : (double)(run - view_pre[g]);
    } else {
      s_tot = run;
      if (blockIdx.y == 0) counts[g] = (double)run;
    }
  }
  __syncthreads();
  const long long tot = s_tot;
  // fused running-mean update (prototypes.py:158-163; the arithmetic of proto_update_kernel): old count from the snapshot
  float upd_old = 0.f, upd_den = 1.f;
  if (!VIEW && proto) {
    if (count_is_int64) {
      const long long o = (long long)count_snap[g];
      upd_old = (float)o;
      upd_den = (float)(o + tot);
      if (tid == 0 && blockIdx.y == 0 && tot > 0) reinterpret_cast<long long*>(count)[g] = o + tot;
    } else {
      const float o = __uint_as_float((unsigned)count_snap[g]);
      upd_old = o;
      upd_den = __fadd_rn(o, (float)(double)tot);
      if (tid == 0 && blockIdx.y == 0 && tot > 0) reinterpret_cast<float*>(count)[g] = upd_den;
    }
    if (ready && g == 0 && blockIdx.y == 0 && tid < 32) {   // all counts non-zero after the update (prototypes.py:31-40)
      int nz = 1;
      for (int t = tid; t < Tn; t += 32) {
        long long n = 0;
        for (int bb = 0; bb < B; ++bb) n += n_bt[bb * Tn + t];
        bool nonzero;
        if (count_is_int64) {
          const long long o = (long long)count_snap[t];
          nonzero = (n > 0 ? o + n : o) != 0;
        } else {
          const float o = __uint_as_float((unsigned)count_snap[t]);
          nonzero = (n > 0 ? __fadd_rn(o, (float)(double)n) : o) != 0.f;
        }
        nz &= nonzero ? 1 : 0;
      }
      nz = __all_sync(0xffffffffu, nz);
      if (tid == 0) *ready = nz;
    }
  }
  if (gather && mode == 0 && tot > 0)
    for (int bb = tid; bb < B; bb += blockDim.x) {
      s_lo[bb] = (int)(((long long)D * s_pre[bb]) / tot);
      s_hi[bb] = s_nb[bb] > 0 ? (int)(((long long)D * (s_pre[bb] + s_nb[bb]) - 1) / tot) : -2;
    }
  __syncthreads();
  const int rl = tid % kFinRows, bl = tid / kFinRows;
  const int r = blockIdx.y * kFinRows + rl;
  double acc = 0.0;
  if (gather && r < D && tot > 0) {
    if (mode != 0) {
      for (int bb = bl; bb < B; bb += kFinLanes) acc += (double)partial[(((int64_t)bb * D + r) * Tn + g) * 2];
    } else {
      // the kFinLanes threads of a row walk the images together and split the CHANNELS of a contributing image
      // (a row takes ~N_g / n_b channel runs of one or two images): four independent loads in flight per thread,
      // never a serial chain of L2 round trips
      auto ceil_div = [](long long a, long long d) { return a <= 0 ? 0LL : (a + d - 1) / d; };
      auto add_range = [&](int bb, long long lo, long long hi, int part) {
        for (long long c0 = lo + bl; c0 < hi; c0 += 4 * kFinLanes) {
          float v[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const long long c = c0 + k * kFinLanes;
            v[k] = c < hi ? partial[(((int64_t)bb * D + c) * Tn + g) * 2 + part] : 0.f;
          }
#pragma unroll
          for (int k = 0; k < 4; ++k) acc += (double)v[k];
        }
      };
      for (int bb = 0; bb < B; ++bb) {
        const long long nb = s_nb[bb];
        if (nb <= 0 || r < s_lo[bb] || r > s_hi[bb] + 1) continue;
        // channels c with r0(c) == r   <=>  r*tot <= D*pre + c*nb < (r+1)*tot
        const long long off = (long long)D * s_pre[bb];
        long long c_lo, c_hi, d_lo = 0;
        if ((long long)(D + 1) * tot < 0x7fffffffLL) {   // everything fits 32 bits: cheap divisions
          auto cd32 = [](long long a, unsigned d) { return a <= 0 ? 0LL : (long long)(((unsigned)a + d - 1u) / d); };
          c_lo = cd32((long long)r * tot - off, (unsigned)nb);
          c_hi = cd32((long long)(r + 1) * tot - off, (unsigned)nb);
          if (r > 0) d_lo = cd32((long long)(r - 1) * tot - off, (unsigned)nb);
        } else {
          c_lo = ceil_div((long long)r * tot - off, nb);
          c_hi = ceil_div((long long)(r + 1) * tot - off, nb);
          if (r > 0) d_lo = ceil_div((long long)(r - 1) * tot - off, nb);
        }
        if (c_hi > D) c_hi = D;
        add_range(bb, c_lo, c_hi, 0);
        // channels with r0(c) == r - 1 contribute their high part
        if (r > 0) add_range(bb, d_lo, c_lo > D ? D : c_lo, 1);
      }
    }
  }
  s_red[bl][rl] = acc;
  __syncthreads();
  if (bl == 0 && r < D) {
    double t = 0.0;
    if (gather) {
#pragma unroll
      for (int i = 0; i < kFinLanes; ++i) t += s_red[i][rl];  // fixed order: deterministic
      sums[(int64_t)g * D + r] = t;
    } else {
      t = sums[(int64_t)g * D + r];  // the accumulate launch has already added every image into the row
    }
    if (!VIEW && proto && tot > 0) {
      const int64_t i = (int64_t)g * D + r;
      proto[i] = __fdiv_rn(__fadd_rn((float)t, __fmul_rn(upd_old, proto[i])), upd_den);
    }
  }
}

// Count exchange without peer memory: this rank's task totals (the payload of the all-gather), then the view of rank
// `rank` from the gathered [world][Tn] table, summed in rank order.
__global__ void __launch_bounds__(kMaxTasks) proto_task_totals_kernel(const int32_t* __restrict__ n_bt, int B, int Tn,
                                                                     long long* __restrict__ totals) {
  pdl_wait();
  pdl_trigger();
  const int t = threadIdx.x;
  if (t >= Tn) return;
  long long n = 0;
  for (int bb = 0; bb < B; ++bb) n += n_bt[bb * Tn + t];
  totals[t] = n;
}

__global__ void __launch_bounds__(kMaxTasks) proto_count_view_kernel(const long long* __restrict__ table, int world,
                                                                    int rank, int Tn, long long* __restrict__ view_pre,
                                                                    long long* __restrict__ view_n) {
  pdl_wait();
  pdl_trigger();
  const int t = threadIdx.x;
  if (t >= Tn) return;
  long long pre = 0, n = 0;
  for (int r = 0; r < world; ++r) {
    const long long v = table[(int64_t)r * Tn + t];
    if (r < rank) pre += v;
    n += v;
  }
  view_pre[t] = pre;
  view_n[t] = n;
}

// proto[g] = (S[g] + cnt[g]*proto[g]) / (cnt[g] + N[g]), cnt[g] += N[g]; separate fp32
// roundings per operation (torch evaluates them as separate kernels).  TCAP: task capacity of the shared arrays.
template <int TCAP>
__global__ void __launch_bounds__(512) proto_update_kernel(float* __restrict__ proto, void* __restrict__ count,
                                                           int count_is_int64, const double* __restrict__ sums,
                                                           const double* __restrict__ counts, int Tn, int D,
                                                           int32_t* __restrict__ ready) {
  __shared__ float s_old[TCAP], s_den[TCAP];
  __shared__ int s_upd[TCAP];
  __shared__ int s_nonzero;
  if (threadIdx.x == 0) s_nonzero = 0;
  pdl_wait();
  pdl_trigger();
  __syncthreads();
  if (threadIdx.x < Tn) {
    const int g = threadIdx.x;
    const double n = counts[g];
    float oldc, den;
    int nz;
    if (count_is_int64) {
      int64_t* c = reinterpret_cast<int64_t*>(count);
      const int64_t o = c[g];
      const int64_t nn = o + (int64_t)n;
      oldc = (float)o;
      den = (float)nn;
      if (n > 0) c[g] = nn;
      nz = (n > 0 ? nn : o) != 0;
    } else {
      float* c = reinterpret_cast<float*>(count);
      const float o = c[g];
      const float nn = __fadd_rn(o, (float)n);
      oldc = o;
      den = nn;
      if (n > 0) c[g] = nn;
      nz = (n > 0 ? nn : o) != 0.f;
    }
    s_old[g] = oldc;
    s_den[g] = den;
    s_upd[g] = n > 0;
    if (nz) atomicAdd(&s_nonzero, 1);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < Tn * D; i += blockDim.x) {
    const int g = i / D;
    if (s_upd[g]) {
      const float num = __fadd_rn((float)sums[i], __fmul_rn(s_old[g], proto[i]));
      proto[i] = __fdiv_rn(num, s_den[g]);
    }
  }
  if (threadIdx.x == 0 && ready) *ready = (s_nonzero == Tn) ? 1 : 0;
}

}  // namespace bacs

using namespace bacs;

extern "C" {

size_t bacs_proto_workspace_bytes(int B, int D, int T) {
  // partial sums | snapshot of the counts (8 bytes per task)
  return align_up((size_t)B * D * T * 2 * sizeof(float), 256) + align_up((size_t)T * 8, 256);
}

static int proto_accumulate_impl(const void* features, int dtype, int B, int D, int h, int w, const int8_t* task,
                                 const int32_t* rank, const int32_t* n_bt, int T, int mode, double* sums, double* counts,
                                 void* workspace, size_t workspace_bytes, float* proto, void* count, int count_is_int64,
                                 int32_t* ready, const long long* view_pre, const long long* view_n,
                                 bacs_stream_t stream) {
  BACS_REQUIRE(features && task && rank && n_bt && sums && counts && workspace, "bacs_proto_accumulate: null pointer");
  BACS_REQUIRE(B > 0 && D > 0 && h > 0 && w > 0 && B <= kFinMaxB, "bacs_proto_accumulate: bad shape (B <= 1024)");
  BACS_REQUIRE(T > 0 && T <= kMaxTasks, "bacs_proto_accumulate: T=%d not in [1,%d]", T, kMaxTasks);
  BACS_REQUIRE(mode == 0 || mode == 1, "bacs_proto_accumulate: mode must be 0 (exact) or 1 (channel)");
  if (workspace_bytes < bacs_proto_workspace_bytes(B, D, T)) {
    set_error("bacs_proto_accumulate: workspace %zu < %zu", workspace_bytes, bacs_proto_workspace_bytes(B, D, T));
    return BACS_ERR_WORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  float* partial = reinterpret_cast<float*>(workspace);
  unsigned long long* snap = proto ? reinterpret_cast<unsigned long long*>(
                                         reinterpret_cast<char*>(workspace) + align_up((size_t)B * D * T * 2 * sizeof(float), 256))
                                   : nullptr;
  const void* count_raw = count;
  const int hw = h * w;
  // more than kTaskWindow tasks: one launch with a grid dimension over 32-task windows (the MANY instantiations), each
  // block with the shared memory of a 32-task launch; the features are read once per window, the later reads from L2
  const bool many = T > kTaskWindow;
  const int n_win = (T + kTaskWindow - 1) / kTaskWindow;
  const int Tw = many ? kTaskWindow : T;
  dim3 grid((D + kAccWarps - 1) / kAccWarps, B, n_win);
  const size_t acc_smem = (size_t)kAccWarps * Tw * 64 * sizeof(float);
  const size_t vec_smem = (size_t)kAccWarps * ((Tw * 2 + 2) * 32 + 33) * sizeof(float);
  const bool vec = hw % 8 == 0 && (reinterpret_cast<uintptr_t>(features) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(task) & 7) == 0 && (reinterpret_cast<uintptr_t>(rank) & 15) == 0;
  // 16-bit features on 32-pixel chunks, 16-channel blocks: one-hot GEMM on the tensor cores (BACS_NO_PROTO_MMA=1: off)
  const bool mma = vec && dtype != BACS_F32 && hw % 32 == 0 && D % 16 == 0 && getenv("BACS_NO_PROTO_MMA") == nullptr;
  const bool view = view_pre != nullptr;   // global view: its own instantiations, the local ones stay as they are
  if (mma) {
    launch_pdl(proto_zero_sums_kernel, dim3((T * D + 255) / 256), dim3(256), 0, s, sums, T * D);
    BACS_CHECK_LAUNCH("bacs_proto_accumulate(zero)");
    dim3 mgrid((D / 16 + kMmaWarps - 1) / kMmaWarps, B, n_win);
    const int nt = (T + 7) / 8;
#define BACS_MMA_LAUNCH(TT, NTV, M)                                                                                     \
  launch_pdl(view ? proto_accumulate_mma_kernel<TT, NTV, M, true> : proto_accumulate_mma_kernel<TT, NTV, M>, mgrid,      \
             dim3(32 * kMmaWarps), 0, s, reinterpret_cast<const TT*>(features), B, D, hw, task, rank, n_bt, T, mode, sums, \
             count_raw, count_is_int64, snap, view_pre, view_n)
#define BACS_MMA_NT(TT)                                 \
  do {                                                  \
    if (many) BACS_MMA_LAUNCH(TT, 4, true);             \
    else if (nt == 1) BACS_MMA_LAUNCH(TT, 1, false);    \
    else if (nt == 2) BACS_MMA_LAUNCH(TT, 2, false);    \
    else if (nt == 3) BACS_MMA_LAUNCH(TT, 3, false);    \
    else BACS_MMA_LAUNCH(TT, 4, false);                 \
  } while (0)
    if (dtype == BACS_BF16) BACS_MMA_NT(__nv_bfloat16);
    else BACS_MMA_NT(__half);
#undef BACS_MMA_NT
#undef BACS_MMA_LAUNCH
  } else {
  BACS_DISPATCH_DTYPE(dtype, TT, {
    // the table of a 32-task window (vec: 68.6 KB, scalar: 64 KB) needs the opt-in above the 48 KB default
    auto kern = view ? (vec ? (many ? proto_accumulate_vec_kernel<TT, true, true> : proto_accumulate_vec_kernel<TT, false, true>)
                            : (many ? proto_accumulate_kernel<TT, true, true> : proto_accumulate_kernel<TT, false, true>))
                     : (vec ? (many ? proto_accumulate_vec_kernel<TT, true> : proto_accumulate_vec_kernel<TT>)
                            : (many ? proto_accumulate_kernel<TT, true> : proto_accumulate_kernel<TT>));
    const size_t smem = vec ? vec_smem : acc_smem;
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) {
        set_error("bacs_proto_accumulate: shared memory opt-in failed: %s", cudaGetErrorString(e));
        return BACS_ERR_CUDA;
      }
    }
    launch_pdl(kern, grid, dim3(32 * kAccWarps), smem, s, reinterpret_cast<const TT*>(features), B, D, hw, task, rank,
               n_bt, T, mode, partial, count_raw, count_is_int64, snap, view_pre, view_n);
  });
  }
  BACS_CHECK_LAUNCH("bacs_proto_accumulate");
  launch_pdl(view ? proto_finalize_kernel<true> : proto_finalize_kernel<>, dim3(T, (D + kFinRows - 1) / kFinRows),
             dim3(kFinRows * kFinLanes), 0, s, partial, B, D, n_bt, T, mode, sums, counts, proto, count, count_is_int64,
             (const unsigned long long*)snap, ready, mma ? 0 : 1, view_pre, view_n);
  BACS_CHECK_LAUNCH("bacs_proto_accumulate(finalize)");
  return BACS_OK;
}

int bacs_proto_accumulate(const void* features, int dtype, int B, int D, int h, int w, const int8_t* task,
                          const int32_t* rank, const int32_t* n_bt, int T, int mode, double* sums, double* counts,
                          void* workspace, size_t workspace_bytes, bacs_stream_t stream) {
  return proto_accumulate_impl(features, dtype, B, D, h, w, task, rank, n_bt, T, mode, sums, counts, workspace,
                               workspace_bytes, nullptr, nullptr, 0, nullptr, nullptr, nullptr, stream);
}

int bacs_proto_accumulate_view(const void* features, int dtype, int B, int D, int h, int w, const int8_t* task,
                               const int32_t* rank, const int32_t* n_bt, int T, int mode, const int64_t* view_pre,
                               const int64_t* view_n, double* sums, double* counts, void* workspace,
                               size_t workspace_bytes, bacs_stream_t stream) {
  BACS_REQUIRE((view_pre == nullptr) == (view_n == nullptr), "bacs_proto_accumulate_view: view_pre and view_n go together");
  BACS_REQUIRE(T > 0 && T <= kMaxTasks, "bacs_proto_accumulate_view: T=%d not in [1,%d]", T, kMaxTasks);
  BACS_REQUIRE(view_pre == nullptr || mode == 0, "bacs_proto_accumulate_view: a view needs mode 0 (exact)");
  return proto_accumulate_impl(features, dtype, B, D, h, w, task, rank, n_bt, T, mode, sums, counts, workspace,
                               workspace_bytes, nullptr, nullptr, 0, nullptr, reinterpret_cast<const long long*>(view_pre),
                               reinterpret_cast<const long long*>(view_n), stream);
}

int bacs_proto_task_totals(const int32_t* n_bt, int B, int T, int64_t* totals, bacs_stream_t stream) {
  BACS_REQUIRE(n_bt && totals, "bacs_proto_task_totals: null pointer");
  BACS_REQUIRE(B > 0, "bacs_proto_task_totals: bad shape");
  BACS_REQUIRE(T > 0 && T <= kMaxTasks, "bacs_proto_task_totals: T=%d not in [1,%d]", T, kMaxTasks);
  launch_pdl(proto_task_totals_kernel, dim3(1), dim3(kMaxTasks), 0, (cudaStream_t)stream, n_bt, B, T,
             reinterpret_cast<long long*>(totals));
  BACS_CHECK_LAUNCH("bacs_proto_task_totals");
  return BACS_OK;
}

int bacs_proto_count_view(const int64_t* table, int world, int rank, int T, int64_t* view_pre, int64_t* view_n,
                          bacs_stream_t stream) {
  BACS_REQUIRE(table && view_pre && view_n, "bacs_proto_count_view: null pointer");
  BACS_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bacs_proto_count_view: bad rank/world");
  BACS_REQUIRE(T > 0 && T <= kMaxTasks, "bacs_proto_count_view: T=%d not in [1,%d]", T, kMaxTasks);
  launch_pdl(proto_count_view_kernel, dim3(1), dim3(kMaxTasks), 0, (cudaStream_t)stream,
             reinterpret_cast<const long long*>(table), world, rank, T, reinterpret_cast<long long*>(view_pre),
             reinterpret_cast<long long*>(view_n));
  BACS_CHECK_LAUNCH("bacs_proto_count_view");
  return BACS_OK;
}

int bacs_proto_accumulate_update(const void* features, int dtype, int B, int D, int h, int w, const int8_t* task,
                                 const int32_t* rank, const int32_t* n_bt, int T, int mode, double* sums, double* counts,
                                 void* workspace, size_t workspace_bytes, float* proto, void* count, int count_is_int64,
                                 int32_t* ready, bacs_stream_t stream) {
  BACS_REQUIRE(proto && count, "bacs_proto_accumulate_update: null pointer");
  BACS_REQUIRE(T > 0 && T <= kMaxTasks, "bacs_proto_accumulate_update: T=%d not in [1,%d]", T, kMaxTasks);
  return proto_accumulate_impl(features, dtype, B, D, h, w, task, rank, n_bt, T, mode, sums, counts, workspace,
                               workspace_bytes, proto, count, count_is_int64, ready, nullptr, nullptr, stream);
}

int bacs_proto_update(float* proto, void* count, int count_is_int64, const double* sums, const double* counts, int T,
                      int D, int32_t* ready, bacs_stream_t stream) {
  BACS_REQUIRE(proto && count && sums && counts, "bacs_proto_update: null pointer");
  BACS_REQUIRE(D > 0, "bacs_proto_update: bad shape");
  BACS_REQUIRE(T > 0 && T <= kMaxTasks, "bacs_proto_update: T=%d not in [1,%d]", T, kMaxTasks);
  launch_pdl(T <= 64 ? proto_update_kernel<64> : proto_update_kernel<kMaxTasks>, dim3(1), dim3(512), 0, (cudaStream_t)stream, proto, count, count_is_int64, sums, counts, T, D,
             ready);
  BACS_CHECK_LAUNCH("bacs_proto_update");
  return BACS_OK;
}

}  // extern "C"
