// Cross-GPU combination of the per-step state over NVLink peer memory, fused with the prototype update.
//
// The only cross-rank state of the BACS loss path is a few tens of KB per step (per-task feature sums and
// pixel counts; the confusion matrix at evaluation): latency-bound, so instead of a ring / tree collective every
// rank reads all peers' buffers directly ("one-shot" all-reduce) and applies the running-mean update
// (loss/prototypes.py:158-163) in the same launch:
//   1. copy my packed fp64 state into my slot of the symmetric buffer (double-buffered by step parity),
//   2. publish: fence.sys + release-store of the step number into every peer's flag row,
//   3. wait until every peer's flag for me shows this step (acquire loads; the spin is bounded in wall-clock time
//      (bacs_peer_set_timeout_ms, default 30 s) so a missing rank can never hang the GPU for good),
//   4. sum the W peer buffers in RANK ORDER (bit-identical result on every rank), write it back to `packed`,
//   5. (optional) proto[g] = (S[g] + cnt[g] proto[g]) / (cnt[g] + N[g]), cnt[g] += N[g]; ready flag.
// On a time-out NOTHING is combined: `packed`, the prototypes and the counts keep their values, the sticky error
// word receives the step number and the ready flag is cleared; the host raises at its next check
// (distributed.PeerReducer.check).  A rank never applies a sum that may contain a stale or half-written peer slot.
// A peer can only be one step ahead (it needs my flag of step e+1 to finish step e+1), and it then writes the
// OTHER parity slot, so reads of step e never race with writes of step e+1.
//
// Count phase (global view of the exact-mode prototype sums, before the accumulate launch): every rank pushes its
// task totals sum_b n_bt[b][t] into row `rank` of every peer's count table (double-buffered by the parity of a step
// counter of its own), publishes with a release-store into the peers' count-flag rows (apart from the flags of the sums
// phase), waits for every peer as above, then sums its local table in rank order into view_pre (ranks below) and view_n
// (all ranks).  On a time-out the view is marked invalid (view_n = -1): the accumulate launch then adds nothing and
// writes -inf counts, so the running-mean update that follows leaves every prototype and count untouched on this rank
// (and on every rank that combines its state); the sticky error word receives the count step as above.
#include "common.cuh"

namespace bacs {

constexpr int kPeerMaxWorld = 16;
struct PeerPtrs {
  double* buf[kPeerMaxWorld];         // peer r's symmetric region: [2][n_max] doubles
  unsigned int* flag[kPeerMaxWorld];  // peer r's flag row: [kPeerMaxWorld] step numbers, one per source rank
};

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ double ld_relaxed_sys_f64(const double* p) {
  double v;
  asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

static unsigned long long g_peer_timeout_ns = 30ull * 1000ull * 1000ull * 1000ull;

// TCAP: task capacity of the fused update's shared arrays (64 up to 64 tasks, kMaxTasks above).
template <int TCAP>
__global__ void __launch_bounds__(1024) peer_allreduce_update_kernel(PeerPtrs pp, int rank, int world, int n, int n_max,
                                                                     unsigned long long timeout_ns,
                                                                     double* __restrict__ packed,
                                                                     unsigned int* __restrict__ step_dev,
                                                                     int* __restrict__ error_dev,
                                                                     // optional fused prototype update
                                                                     float* __restrict__ proto, void* __restrict__ count,
                                                                     int count_is_int64, int Tn, int D,
                                                                     int32_t* __restrict__ ready) {
  __shared__ int s_timeout;
  pdl_wait();     // `packed` comes from the launches before this one; the launch itself overlaps their tail
  pdl_trigger();  // the next launch (seen heads) may become resident; it waits for this grid's completion itself
  const unsigned int step = *step_dev + 1u;
  const int slot = (int)(step & 1u);
  double* mine = pp.buf[rank] + (size_t)slot * n_max;
  if (threadIdx.x == 0) s_timeout = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) mine[i] = packed[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x < world) {
    st_release_sys(pp.flag[threadIdx.x] + rank, step);  // tell peer threadIdx.x that my slot is filled
    // wait for that peer's slot (bounded: a missing peer must not hang the GPU)
    const unsigned int* f = pp.flag[rank] + threadIdx.x;
    const unsigned long long t0 = global_timer_ns();
    unsigned int polls = 0;
    while ((int)(ld_acquire_sys(f) - step) < 0) {
      if ((++polls & 1023u) == 0 && global_timer_ns() - t0 > timeout_ns) {
        s_timeout = 1;
        break;
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) *step_dev = step;  // the step counter advances either way (flags stay monotonic)
  if (s_timeout) {  // uniform: leave every output untouched, report, and let the host raise
    if (threadIdx.x == 0) {
      if (error_dev) *error_dev = (int)step;
      if (ready) *ready = 0;
    }
    return;
  }
  // every peer value of two elements of a thread is requested before the first add: one NVLink round trip per pair of
  // elements instead of one per (element, peer) -- the loads are volatile asm and are not hoisted above the adds otherwise
  for (int i0 = threadIdx.x; i0 < n; i0 += 2 * blockDim.x) {
    const int i1 = i0 + blockDim.x;
    double s0 = 0.0, s1 = 0.0;
    for (int rg = 0; rg < world; rg += 8) {  // eight peers at a time (registers), rank order: bit-identical on every rank
      double v0[8], v1[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        v0[k] = v1[k] = 0.0;
        if (rg + k < world) {
          v0[k] = ld_relaxed_sys_f64(pp.buf[rg + k] + (size_t)slot * n_max + i0);
          if (i1 < n) v1[k] = ld_relaxed_sys_f64(pp.buf[rg + k] + (size_t)slot * n_max + i1);
        }
      }
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (rg + k < world) {
          s0 += v0[k];
          s1 += v1[k];
        }
    }
    packed[i0] = s0;
    if (i1 < n) packed[i1] = s1;
  }
  if (proto == nullptr) return;
  __syncthreads();  // packed[] (global, this block) is complete
  // ---- fused running-mean update (same arithmetic as proto_update_kernel) ----
  __shared__ float s_old[TCAP], s_den[TCAP];
  __shared__ int s_upd[TCAP];
  __shared__ int s_nonzero;
  const double* sums = packed;
  const double* counts = packed + (size_t)Tn * D;
  if (threadIdx.x == 0) s_nonzero = 0;
  __syncthreads();
  if (threadIdx.x < Tn) {
    const int g = threadIdx.x;
    const double nn_d = counts[g];
    float oldc, den;
    int nz;
    if (count_is_int64) {
      int64_t* c = reinterpret_cast<int64_t*>(count);
      const int64_t o = c[g];
      const int64_t nn = o + (int64_t)nn_d;
      oldc = (float)o;
      den = (float)nn;
      if (nn_d > 0) c[g] = nn;
      nz = (nn_d > 0 ? nn : o) != 0;
    } else {
      float* c = reinterpret_cast<float*>(count);
      const float o = c[g];
      const float nn = __fadd_rn(o, (float)nn_d);
      oldc = o;
      den = nn;
      if (nn_d > 0) c[g] = nn;
      nz = (nn_d > 0 ? nn : o) != 0.f;
    }
    s_old[g] = oldc;
    s_den[g] = den;
    s_upd[g] = nn_d > 0;
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

__global__ void __launch_bounds__(kMaxTasks) peer_count_exchange_kernel(PeerPtrs pp, int rank, int world,
                                                                       unsigned long long timeout_ns,
                                                                       const int32_t* __restrict__ n_bt, int B, int Tn,
                                                                       unsigned int* __restrict__ step_dev,
                                                                       int* __restrict__ error_dev,
                                                                       long long* __restrict__ view_pre,
                                                                       long long* __restrict__ view_n) {
  __shared__ long long s_tot[kMaxTasks];
  __shared__ int s_timeout;
  pdl_wait();     // n_bt comes from the task down-sample
  pdl_trigger();  // the accumulate launch waits for this grid's completion itself
  const unsigned int step = *step_dev + 1u;
  const size_t slot = (size_t)(step & 1u) * world * kMaxTasks;   // table: [2][world][kMaxTasks] int64 per rank
  if (threadIdx.x == 0) s_timeout = 0;
  if (threadIdx.x < Tn) {
    long long n = 0;
    for (int bb = 0; bb < B; ++bb) n += n_bt[bb * Tn + threadIdx.x];
    s_tot[threadIdx.x] = n;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < world * Tn; i += blockDim.x) {
    const int r = i / Tn, t = i - r * Tn;
    reinterpret_cast<long long*>(pp.buf[r])[slot + (size_t)rank * kMaxTasks + t] = s_tot[t];
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x < world) {
    st_release_sys(pp.flag[threadIdx.x] + rank, step);
    const unsigned int* f = pp.flag[rank] + threadIdx.x;
    const unsigned long long t0 = global_timer_ns();
    unsigned int polls = 0;
    while ((int)(ld_acquire_sys(f) - step) < 0) {
      if ((++polls & 1023u) == 0 && global_timer_ns() - t0 > timeout_ns) {
        s_timeout = 1;
        break;
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) *step_dev = step;
  if (threadIdx.x >= Tn) return;
  const int t = threadIdx.x;
  if (s_timeout) {
    if (t == 0 && error_dev) *error_dev = (int)step;
    view_pre[t] = 0;
    view_n[t] = -1;
    return;
  }
  const double* mine = pp.buf[rank] + slot + t;
  long long pre = 0, n = 0;
  for (int r = 0; r < world; ++r) {   // rank order: the images of rank r come after those of ranks 0 .. r-1
    const long long v = __double_as_longlong(ld_relaxed_sys_f64(mine + (size_t)r * kMaxTasks));
    if (r < rank) pre += v;
    n += v;
  }
  view_pre[t] = pre;
  view_n[t] = n;
}

}  // namespace bacs

using namespace bacs;

extern "C" {

int bacs_peer_count_exchange(const int32_t* n_bt, int B, int T, int rank, int world, const uint64_t* peer_table_host,
                             const uint64_t* peer_flag_host, uint32_t* step_dev, int32_t* error_dev, int64_t* view_pre,
                             int64_t* view_n, bacs_stream_t stream) {
  BACS_REQUIRE(n_bt && peer_table_host && peer_flag_host && step_dev && view_pre && view_n,
               "bacs_peer_count_exchange: null pointer");
  BACS_REQUIRE(world >= 1 && world <= kPeerMaxWorld && rank >= 0 && rank < world, "bacs_peer_count_exchange: bad rank/world");
  BACS_REQUIRE(B > 0, "bacs_peer_count_exchange: bad shape");
  BACS_REQUIRE(T > 0 && T <= kMaxTasks, "bacs_peer_count_exchange: T=%d not in [1,%d]", T, kMaxTasks);
  PeerPtrs pp;
  for (int r = 0; r < kPeerMaxWorld; ++r) {
    pp.buf[r] = r < world ? reinterpret_cast<double*>(peer_table_host[r]) : nullptr;
    pp.flag[r] = r < world ? reinterpret_cast<unsigned int*>(peer_flag_host[r]) : nullptr;
  }
  launch_pdl(peer_count_exchange_kernel, dim3(1), dim3(kMaxTasks), 0, (cudaStream_t)stream, pp, rank, world,
             g_peer_timeout_ns, n_bt, B, T, step_dev, error_dev, reinterpret_cast<long long*>(view_pre),
             reinterpret_cast<long long*>(view_n));
  BACS_CHECK_LAUNCH("bacs_peer_count_exchange");
  return BACS_OK;
}

int bacs_peer_set_timeout_ms(int64_t ms) {
  BACS_REQUIRE(ms > 0, "bacs_peer_set_timeout_ms: the time-out must be positive");
  g_peer_timeout_ns = (unsigned long long)ms * 1000000ull;
  return BACS_OK;
}

int bacs_peer_allreduce(double* packed, int n, int n_max, int rank, int world, const uint64_t* peer_buf_host,
                        const uint64_t* peer_flag_host, uint32_t* step_dev, int32_t* error_dev, float* proto,
                        void* count, int count_is_int64, int T, int D, int32_t* ready, bacs_stream_t stream) {
  BACS_REQUIRE(packed && peer_buf_host && peer_flag_host && step_dev, "bacs_peer_allreduce: null pointer");
  BACS_REQUIRE(world >= 1 && world <= kPeerMaxWorld && rank >= 0 && rank < world, "bacs_peer_allreduce: bad rank/world");
  BACS_REQUIRE(n > 0 && n <= n_max, "bacs_peer_allreduce: n=%d exceeds the symmetric buffer (%d)", n, n_max);
  if (proto) {
    BACS_REQUIRE(count && D > 0 && n >= T * D + T, "bacs_peer_allreduce: bad prototype shape");
    BACS_REQUIRE(T > 0 && T <= kMaxTasks, "bacs_peer_allreduce: T=%d not in [1,%d]", T, kMaxTasks);
  }
  PeerPtrs pp;
  for (int r = 0; r < kPeerMaxWorld; ++r) {
    pp.buf[r] = r < world ? reinterpret_cast<double*>(peer_buf_host[r]) : nullptr;
    pp.flag[r] = r < world ? reinterpret_cast<unsigned int*>(peer_flag_host[r]) : nullptr;
  }
  launch_pdl(proto && T > 64 ? peer_allreduce_update_kernel<kMaxTasks> : peer_allreduce_update_kernel<64>, dim3(1),
             dim3(1024), 0, (cudaStream_t)stream, pp, rank, world, n, n_max, g_peer_timeout_ns, packed, step_dev,
             error_dev, proto, count, count_is_int64, T, D, ready);
  BACS_CHECK_LAUNCH("bacs_peer_allreduce");
  return BACS_OK;
}

}  // extern "C"
