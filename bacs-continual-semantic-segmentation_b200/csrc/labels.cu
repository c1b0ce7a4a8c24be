// Label kernels: histogram, continual-learning remap, nearest down-sample + task / rank.
#include <stdarg.h>
#include <limits.h>

#include <algorithm>

#include "common.cuh"

namespace bacs {

unsigned long long g_launch_count = 0;
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// -------------------------------------------------------------------------------------
// Histogram of int64 labels.  Each thread walks 16-byte pairs with a run-length
// accumulator so that the (typical) long runs of one label cost one shared atomic.
// -------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) label_hist_kernel(const int64_t* __restrict__ labels, int64_t n,
                                                         unsigned long long* __restrict__ hist) {
  __shared__ unsigned int sh[257];
  for (int i = threadIdx.x; i < 257; i += blockDim.x) sh[i] = 0;
  __syncthreads();
  // each thread owns contiguous chunks of 8 labels; chunks are strided over the grid
  const int64_t nchunk = (n + 7) >> 3;
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < nchunk;
       c += (int64_t)gridDim.x * blockDim.x) {
    const int64_t base = c << 3;
    int cur = -1;
    unsigned int run = 0;
    if (base + 8 <= n) {
      const longlong2* p = reinterpret_cast<const longlong2*>(labels + base);
      longlong2 v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) v[k] = __ldg(p + k);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int64_t l = (k & 1) ? v[k >> 1].y : v[k >> 1].x;
        const int bin = (l >= 0 && l < 256) ? (int)l : 256;
        if (bin == cur) {
          ++run;
        } else {
          if (run) atomicAdd(&sh[cur], run);
          cur = bin;
          run = 1;
        }
      }
    } else {
      for (int64_t i = base; i < n; ++i) {
        const int64_t l = labels[i];
        const int bin = (l >= 0 && l < 256) ? (int)l : 256;
        if (bin == cur) {
          ++run;
        } else {
          if (run) atomicAdd(&sh[cur], run);
          cur = bin;
          run = 1;
        }
      }
    }
    if (run) atomicAdd(&sh[cur], run);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 257; i += blockDim.x)
    if (sh[i]) atomicAdd(&hist[i], (unsigned long long)sh[i]);
}

// -------------------------------------------------------------------------------------
// Remap.  Domain of values: [lo, lo + n_dom), n_dom <= 1024.
// -------------------------------------------------------------------------------------
constexpr int kMaxDom = 1024;
constexpr int kPresStride = kMaxDom + 8;  // [0,kMaxDom) presence flags, then: below-domain, above-domain present

__global__ void __launch_bounds__(256) remap_presence_kernel(const int64_t* __restrict__ in, int64_t ppi, int lo,
                                                             int n_dom, int32_t* __restrict__ presence) {
  __shared__ int sh[kPresStride];
  const int img = blockIdx.y;
  for (int i = threadIdx.x; i < kPresStride; i += blockDim.x) sh[i] = 0;
  __syncthreads();
  const int64_t* src = in + (int64_t)img * ppi;
  int last = INT_MIN;
  auto mark = [&](int64_t l) {
    const int64_t r = l - lo;
    const int slot = r < 0 ? kMaxDom : (r >= n_dom ? kMaxDom + 1 : (int)r);
    if (slot != last) {
      sh[slot] = 1;
      last = slot;
    }
  };
  if ((ppi & 1) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
    // 16-byte loads, four in flight per thread
    const longlong2* v = reinterpret_cast<const longlong2*>(src);
    const int64_t nv = ppi >> 1, step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += 4 * step) {
      longlong2 x[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) x[u] = (i + u * step < nv) ? __ldg(v + i + u * step) : make_longlong2(lo, lo);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        mark(x[u].x);
        mark(x[u].y);
      }
    }
  } else {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ppi; i += (int64_t)gridDim.x * blockDim.x)
      mark(src[i]);
  }
  __syncthreads();
  int32_t* pres = presence + (int64_t)img * kPresStride;
  for (int i = threadIdx.x; i < kPresStride; i += blockDim.x)
    if (sh[i]) pres[i] = 1;
}

// Closed form of the sequential in-place remap (training/utils.py:240-248): the labels
// present at entry are visited in ascending order, so a pixel follows v -> f(v) again
// whenever the image is a larger value that was itself present at entry.
__device__ __forceinline__ int chase(int v, const int* map, const int* present, int lo, int n_dom, int masking) {
  int cur = v;
  for (int it = 0; it <= kMaxDom; ++it) {
    const int r = cur - lo;
    const int nxt = (r >= 0 && r < n_dom) ? map[r] : masking;
    const int rn = nxt - lo;
    if (nxt > cur && rn >= 0 && rn < n_dom && present[rn]) {
      cur = nxt;
      continue;
    }
    return nxt;
  }
  return cur;
}

__global__ void __launch_bounds__(256) remap_apply_kernel(const int64_t* __restrict__ in, int64_t* __restrict__ out,
                                                          int64_t ppi, int lo, int n_dom,
                                                          const int32_t* __restrict__ map1, int masking1,
                                                          const int32_t* __restrict__ map2, int masking2,
                                                          const int32_t* __restrict__ presence) {
  __shared__ int m1[kMaxDom], m2[kMaxDom], p1[kMaxDom], p2[kMaxDom], lut[kMaxDom];
  __shared__ int oob_final[2];
  const int img = blockIdx.y;
  const int32_t* pres = presence + (int64_t)img * kPresStride;
  for (int i = threadIdx.x; i < n_dom; i += blockDim.x) {
    m1[i] = map1[i];
    m2[i] = map2 ? map2[i] : 0;
    p1[i] = pres[i];
    p2[i] = 0;
  }
  __syncthreads();
  const int low_present = pres[kMaxDom], high_present = pres[kMaxDom + 1];
  for (int i = threadIdx.x; i < n_dom; i += blockDim.x) lut[i] = chase(i + lo, m1, p1, lo, n_dom, masking1);
  // out-of-domain values: unmapped -> masking1, chased again if masking1 is larger and present
  const int low1 = chase(lo - 1, m1, p1, lo, n_dom, masking1);
  const int high1 = chase(lo + n_dom, m1, p1, lo, n_dom, masking1);
  __syncthreads();
  if (map2) {
    for (int i = threadIdx.x; i < n_dom; i += blockDim.x)
      if (p1[i]) p2[lut[i] - lo] = 1;
    if (threadIdx.x == 0) {
      if (low_present) p2[low1 - lo] = 1;
      if (high_present) p2[high1 - lo] = 1;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_dom; i += blockDim.x) m1[i] = chase(lut[i], m2, p2, lo, n_dom, masking2);
    if (threadIdx.x == 0) {
      oob_final[0] = chase(low1, m2, p2, lo, n_dom, masking2);
      oob_final[1] = chase(high1, m2, p2, lo, n_dom, masking2);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_dom; i += blockDim.x) lut[i] = m1[i];
  } else if (threadIdx.x == 0) {
    oob_final[0] = low1;
    oob_final[1] = high1;
  }
  __syncthreads();
  const int64_t* src = in + (int64_t)img * ppi;
  int64_t* dst = out + (int64_t)img * ppi;
  auto look = [&](int64_t l) -> int64_t {
    const int64_t r = l - lo;
    return r < 0 ? (int64_t)oob_final[0] : (r >= n_dom ? (int64_t)oob_final[1] : (int64_t)lut[r]);
  };
  if ((ppi & 1) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
    const longlong2* v = reinterpret_cast<const longlong2*>(src);
    longlong2* o = reinterpret_cast<longlong2*>(dst);
    const int64_t nv = ppi >> 1, step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += 4 * step) {
      longlong2 x[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i + u * step < nv) x[u] = __ldg(v + i + u * step);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i + u * step < nv) o[i + u * step] = make_longlong2(look(x[u].x), look(x[u].y));
    }
  } else {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ppi; i += (int64_t)gridDim.x * blockDim.x)
      dst[i] = look(src[i]);
  }
}

// -------------------------------------------------------------------------------------
// Nearest down-sample + task id + raster rank inside (image, task).
// One block per image; pixels are processed in raster order in chunks of blockDim.
// -------------------------------------------------------------------------------------
// KMAX is the task capacity of the per-warp counters: 32 up to 32 tasks, kMaxTasks above.

template <int KMAX>
__global__ void __launch_bounds__(1024) downsample_task_kernel(const int64_t* __restrict__ labels, int H, int W, int h,
                                                               int w, float sy, float sx,
                                                               const int32_t* __restrict__ task_lut, int T,
                                                               int64_t* __restrict__ labels_down,
                                                               int8_t* __restrict__ task, int32_t* __restrict__ rank,
                                                               int32_t* __restrict__ n_bt) {
  __shared__ int lut[256];
  __shared__ int warp_cnt[32][KMAX + 1];
  __shared__ int base[KMAX];
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nwarp = blockDim.x >> 5;
  if (tid < KMAX) base[tid] = 0;
  pdl_wait();
  pdl_trigger();
  for (int i = tid; i < 256; i += blockDim.x) lut[i] = task_lut[i];
  __syncthreads();
  const int hw = h * w;
  const int64_t* src = labels + (int64_t)b * H * W;
  for (int q0 = 0; q0 < hw; q0 += blockDim.x) {
    const int q = q0 + tid;
    int t = -1;
    if (q < hw) {
      const int i = q / w, j = q - i * w;
      const int yi = min((int)floorf((float)i * sy), H - 1);
      const int xi = min((int)floorf((float)j * sx), W - 1);
      const int64_t l = __ldg(src + (int64_t)yi * W + xi);
      if (labels_down) labels_down[(int64_t)b * hw + q] = l;
      if (l >= 0 && l < 256) t = lut[(int)l];
      if (t >= T) t = -1;
      task[(int64_t)b * hw + q] = (int8_t)t;
    }
    // intra-warp rank among lanes with the same task
    const unsigned peers = __match_any_sync(0xffffffffu, t);
    const int within = __popc(peers & ((1u << lane) - 1u));
    for (int g = lane; g < T; g += 32) warp_cnt[wid][g] = 0;
    __syncwarp();
    if (t >= 0 && within == 0) warp_cnt[wid][t] = __popc(peers);
    __syncthreads();
    // exclusive prefix over warps, one thread per task
    if (tid < T) {
      int run = base[tid];
      for (int wv = 0; wv < nwarp; ++wv) {
        const int c = warp_cnt[wv][tid];
        warp_cnt[wv][tid] = run;
        run += c;
      }
      base[tid] = run;
    }
    __syncthreads();
    if (q < hw) rank[(int64_t)b * hw + q] = (t >= 0) ? warp_cnt[wid][t] + within : 0;
    __syncthreads();
  }
  if (tid < T) n_bt[b * T + tid] = base[tid];
}

}  // namespace bacs

using namespace bacs;

extern "C" {

int bacs_version(void) { return BACS_VERSION; }
const char* bacs_last_error_string(void) { return bacs::g_err; }
int bacs_device_sm_count(void) { return bacs::sm_count(); }
unsigned long long bacs_launch_count(void) { return bacs::g_launch_count; }

int bacs_label_hist(const int64_t* labels, int64_t n, int64_t* hist, bacs_stream_t stream) {
  if (n == 0) return BACS_OK;
  BACS_REQUIRE(labels && hist && n > 0, "bacs_label_hist: null pointer or negative size");
  BACS_REQUIRE((reinterpret_cast<uintptr_t>(labels) & 15) == 0, "bacs_label_hist: labels must be 16-byte aligned");
  const int64_t nchunk = (n + 7) >> 3;
  int64_t blocks = (nchunk + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  label_hist_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(labels, n,
                                                                        reinterpret_cast<unsigned long long*>(hist));
  BACS_CHECK_LAUNCH("bacs_label_hist");
  return BACS_OK;
}

int bacs_label_remap(const int64_t* in, int64_t* out, int64_t n_images, int64_t pixels_per_image, int lo, int n_dom,
                     const int32_t* map1, int masking1, const int32_t* map2, int masking2, int32_t* workspace,
                     bacs_stream_t stream) {
  BACS_REQUIRE(in && out && map1 && workspace, "bacs_label_remap: null pointer");
  BACS_REQUIRE(n_dom > 0 && n_dom <= kMaxDom, "bacs_label_remap: domain size %d not in (0,%d]", n_dom, kMaxDom);
  BACS_REQUIRE(n_images >= 0 && n_images < 65536 && pixels_per_image >= 0, "bacs_label_remap: bad sizes");
  BACS_REQUIRE(masking1 >= lo && masking1 < lo + n_dom && (!map2 || (masking2 >= lo && masking2 < lo + n_dom)),
               "bacs_label_remap: masking values must lie inside the domain");
  if (n_images == 0 || pixels_per_image == 0) return BACS_OK;
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(workspace, 0, sizeof(int32_t) * kPresStride * n_images, s);
  if (e != cudaSuccess) {
    set_error("bacs_label_remap: memset failed: %s", cudaGetErrorString(e));
    return BACS_ERR_CUDA;
  }
  int64_t bx = (pixels_per_image + 256 * 8 - 1) / (256 * 8);
  const int64_t cap = std::max<int64_t>(1, (int64_t)sm_count() * 8 / n_images);
  if (bx > cap) bx = cap;
  if (bx < 1) bx = 1;
  dim3 grid((unsigned)bx, (unsigned)n_images);
  remap_presence_kernel<<<grid, 256, 0, s>>>(in, pixels_per_image, lo, n_dom, workspace);
  BACS_CHECK_LAUNCH("bacs_label_remap(presence)");
  remap_apply_kernel<<<grid, 256, 0, s>>>(in, out, pixels_per_image, lo, n_dom, map1, masking1, map2, masking2,
                                         workspace);
  BACS_CHECK_LAUNCH("bacs_label_remap(apply)");
  return BACS_OK;
}

size_t bacs_label_remap_workspace_bytes(int64_t n_images) { return sizeof(int32_t) * kPresStride * (size_t)n_images; }

int bacs_label_downsample_task(const int64_t* labels, int B, int H, int W, int h, int w, const int32_t* task_lut,
                               int T, int64_t* labels_down, int8_t* task, int32_t* rank, int32_t* n_bt,
                               bacs_stream_t stream) {
  BACS_REQUIRE(labels && task_lut && task && rank && n_bt, "bacs_label_downsample_task: null pointer");
  BACS_REQUIRE(B > 0 && H > 0 && W > 0 && h > 0 && w > 0, "bacs_label_downsample_task: bad shape");
  BACS_REQUIRE(T > 0 && T <= kMaxTasks, "bacs_label_downsample_task: T=%d not in [1,%d]", T, kMaxTasks);
  const float sy = (float)H / (float)h, sx = (float)W / (float)w;
  launch_pdl(T <= 32 ? downsample_task_kernel<32> : downsample_task_kernel<kMaxTasks>, dim3(B), dim3(1024), 0,
             (cudaStream_t)stream, labels, H, W, h, w, sy, sx, task_lut, T, labels_down, task, rank, n_bt);
  BACS_CHECK_LAUNCH("bacs_label_downsample_task");
  return BACS_OK;
}

}  // extern "C"
