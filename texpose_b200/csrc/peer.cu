// Gradient exchange of the texture-learner step over NVLink peer memory (SURVEY.md 8e), sm_100a.
//
// The training path has exactly one exchange per step: the mean over the ranks of ~1.7 MB of fp32 head + latent
// gradients.  At that size a library allreduce is all latency (launch + protocol + a second launch to average), so the
// exchange is ONE kernel over CUDA-IPC peer windows:
//
//   window (one per rank, cudaMalloc'ed, opened by every peer):  [ header 1 KB | data buffer 0 | data buffer 1 ]
//     header: arrive[16] u32 (slot p = "rank p's gradients of epoch e are in place"), barrier[16] u32 at byte 128
//     (tp_peer_barrier), status u32 at byte 512
//   step e (e = 1, 2, ...), on every rank, on the caller's stream:
//     1. the caller packs its gradients into data buffer e&1 of its OWN window (ordinary local writes);
//     2. CTA 0 publishes: st.release.sys  arrive[rank] = e  into every peer's header (NVLink stores);
//     3. every CTA waits on its LOCAL header until arrive[p] of every peer p has reached e (ld.acquire.sys, bounded by a
//        timeout; on a timeout the status word is set and `out` is filled with NaN);
//     4. every CTA reads its slice of all `world` buffers (own HBM + NVLink peer loads, 16 B vectors, all loads of a
//        slice in flight together), adds them in rank order 0..world-1 and divides by world -> `out` (local).
//   The rank order makes the result bit-identical on every rank and run to run.  Buffers alternate with the epoch's
//   parity: a peer can only start overwriting buffer e&1 at step e+2, and it cannot pass step e+1's wait before this
//   rank has published e+1, which it does after finishing the reads of step e (stream order) -- no trailing barrier.
//
// Device-held epoch (CUDA-graph capturable exchange): the epoch above is a host argument, which a graph capture freezes.
// The header also holds epoch u32 at byte 768 (the window's device epoch, 0 after create) and stage_done u32 at byte 772
// (CTA completion counter of tp_peer_stage, 0 between launches).  The pair tp_peer_stage + tp_peer_allreduce_mean_dev
// replaces step 1 and the epoch argument:
//   1'. tp_peer_stage copies the caller's gradients into buffer (e+1)&1 of the OWN window, e = the device epoch, then the
//       last CTA to finish stores e+1 (every CTA reads e before it counts itself done; no CTA waits for another);
//   2-4. tp_peer_allreduce_mean_dev runs the same kernel body with epoch = the local window's device epoch.
//   Invariants: epochs still count 1, 2, 3, ... identically on every rank (one stage per exchange, on every rank); eager
//   calls and graph replays of the pair advance the same counter, so they interleave freely; the parity argument above is
//   unchanged, since the stage of step e+2 is stream-ordered after this rank's reduce of step e+1; no kernel waits for its
//   own grid.  A window is driven either by host epochs or by its device epoch, never both (they share the arrive slots).
//
// The window is the one driver object the library creates (like a communicator): tp_peer_window_create / _destroy,
// _export / _import / _release are host calls made once at set-up; the per-step call allocates nothing.
#include "common.cuh"
#include "../../include/texpose_b200.h"

namespace {

constexpr int kMaxWorld = 16;
constexpr int64_t kHeaderBytes = 1024;
constexpr int kStatusWord = 128;   // u32 index of the status word inside the header (byte 512)
constexpr int kBarrierSlot0 = 32;  // u32 index of the barrier slots [16] (tp_peer_barrier; separate from the exchange's arrive[16])
constexpr int kEpochWord = 192;    // u32 index of the device epoch (byte 768): tp_peer_stage advances it, _allreduce_mean_dev reads it
constexpr int kStageDone = 193;    // u32 index of tp_peer_stage's CTA completion counter (byte 772)

struct Windows {
  uint8_t* base[kMaxWorld];
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_peer_v4(const float4* p) {   // relaxed.sys: never served from a stale L1 line
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

template <int kWorld>
__device__ __forceinline__ void reduce_slices(const Windows& w, int64_t data_off, int64_t n4, float divisor, float* out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 v[kWorld];
#pragma unroll
    for (int p = 0; p < kWorld; ++p) v[p] = ld_peer_v4(reinterpret_cast<const float4*>(w.base[p] + data_off) + i);
    float4 a = v[0];
#pragma unroll
    for (int p = 1; p < kWorld; ++p) {
      a.x = __fadd_rn(a.x, v[p].x);
      a.y = __fadd_rn(a.y, v[p].y);
      a.z = __fadd_rn(a.z, v[p].z);
      a.w = __fadd_rn(a.w, v[p].w);
    }
    a.x = __fdiv_rn(a.x, divisor);
    a.y = __fdiv_rn(a.y, divisor);
    a.z = __fdiv_rn(a.z, divisor);
    a.w = __fdiv_rn(a.w, divisor);
    reinterpret_cast<float4*>(out)[i] = a;
  }
}

// Steps 2-4 of one exchange; the two kernels below differ only in where `epoch` comes from.
__device__ __forceinline__ void allreduce_mean_body(const Windows& w, int world, int rank, int64_t n4, int64_t cap_bytes,
                                                    uint32_t epoch, float* out, unsigned long long timeout_ns) {
  uint32_t* my_hdr = reinterpret_cast<uint32_t*>(w.base[rank]);
  // 2. publish (one CTA): this rank's buffer of `epoch` was written by earlier work on this stream
  if (blockIdx.x == 0 && threadIdx.x < world) {
    __threadfence_system();
    st_release_sys(reinterpret_cast<uint32_t*>(w.base[threadIdx.x]) + rank, epoch);
  }
  // 3. wait on the local header for every PEER (every CTA).  The own slot is not waited on: this rank's buffer was written
  // by earlier work on this stream, and only CTA 0 publishes it -- waiting for it would make the other CTAs depend on CTA 0
  // being resident, which a grid larger than one wave does not guarantee.
  int failed = 0;
  if (threadIdx.x < world && threadIdx.x != rank) {
    const uint32_t* flag = my_hdr + threadIdx.x;
    const unsigned long long t0 = global_ns();
    while ((int32_t)(ld_acquire_sys(flag) - epoch) < 0) {
      if (global_ns() - t0 > timeout_ns) {
        failed = 1;
        break;
      }
      __nanosleep(64);
    }
  }
  failed = __syncthreads_or(failed);
  if (failed) {
    // a peer never arrived: report through the status word AND poison this CTA's slice of `out` with NaN, so a caller that
    // does not poll tp_peer_status cannot step the optimizer on stale or partially reduced gradients without noticing
    if (threadIdx.x == 0) atomicMax(my_hdr + kStatusWord, epoch);
    const float nan = __int_as_float(0x7fc00000);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride)
      reinterpret_cast<float4*>(out)[i] = make_float4(nan, nan, nan, nan);
    return;
  }
  // 4. reduce in rank order
  const int64_t data_off = kHeaderBytes + (int64_t)(epoch & 1u) * cap_bytes;
  const float d = (float)world;
  switch (world) {
    case 1: reduce_slices<1>(w, data_off, n4, d, out); break;
    case 2: reduce_slices<2>(w, data_off, n4, d, out); break;
    case 3: reduce_slices<3>(w, data_off, n4, d, out); break;
    case 4: reduce_slices<4>(w, data_off, n4, d, out); break;
    case 5: reduce_slices<5>(w, data_off, n4, d, out); break;
    case 6: reduce_slices<6>(w, data_off, n4, d, out); break;
    case 7: reduce_slices<7>(w, data_off, n4, d, out); break;
    case 8: reduce_slices<8>(w, data_off, n4, d, out); break;
    default: {   // 9..16 ranks: two passes of up to 8 would change the summation order between worlds; keep one loop
      const int64_t stride = (int64_t)gridDim.x * blockDim.x;
      for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 a = ld_peer_v4(reinterpret_cast<const float4*>(w.base[0] + data_off) + i);
        for (int p = 1; p < world; ++p) {
          const float4 v = ld_peer_v4(reinterpret_cast<const float4*>(w.base[p] + data_off) + i);
          a.x = __fadd_rn(a.x, v.x);
          a.y = __fadd_rn(a.y, v.y);
          a.z = __fadd_rn(a.z, v.z);
          a.w = __fadd_rn(a.w, v.w);
        }
        a.x = __fdiv_rn(a.x, d);
        a.y = __fdiv_rn(a.y, d);
        a.z = __fdiv_rn(a.z, d);
        a.w = __fdiv_rn(a.w, d);
        reinterpret_cast<float4*>(out)[i] = a;
      }
    }
  }
}

__global__ void __launch_bounds__(256) peer_allreduce_mean_kernel(const Windows w, int world, int rank, int64_t n4, int64_t cap_bytes,
                                                                  uint32_t epoch, float* out, unsigned long long timeout_ns) {
  allreduce_mean_body(w, world, rank, n4, cap_bytes, epoch, out, timeout_ns);
}

// The epoch is the local window's device epoch, stored by the tp_peer_stage launch that precedes this one on the stream
// (kernel boundary: every CTA reads the same value, and nothing writes it while this grid runs).
__global__ void __launch_bounds__(256) peer_allreduce_mean_dev_kernel(const Windows w, int world, int rank, int64_t n4,
                                                                      int64_t cap_bytes, float* out, unsigned long long timeout_ns) {
  const uint32_t epoch = *(reinterpret_cast<const volatile uint32_t*>(w.base[rank]) + kEpochWord);
  allreduce_mean_body(w, world, rank, n4, cap_bytes, epoch, out, timeout_ns);
}

// Step 1': src[0:n] -> data buffer (e+1)&1 of the local window, then the device epoch becomes e+1.  Every CTA reads e once,
// before it counts itself done; the last CTA to count itself done stores e+1 and re-arms the counter.  No CTA waits.
__global__ void __launch_bounds__(256) peer_stage_kernel(uint8_t* win, int64_t n_floats, int64_t cap_bytes, const float* src) {
  uint32_t* hdr = reinterpret_cast<uint32_t*>(win);
  __shared__ uint32_t e_s;
  if (threadIdx.x == 0) e_s = *reinterpret_cast<volatile uint32_t*>(hdr + kEpochWord);
  __syncthreads();
  const uint32_t e = e_s;
  float* dst = reinterpret_cast<float*>(win + kHeaderBytes + (int64_t)((e + 1u) & 1u) * cap_bytes);
  const int64_t n4 = n_floats / 4;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t i = tid; i < n4; i += stride) reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(src)[i];
  if (tid < n_floats - n4 * 4) dst[n4 * 4 + tid] = src[n4 * 4 + tid];
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(hdr + kStageDone, 1u) == gridDim.x - 1) {
      *reinterpret_cast<volatile uint32_t*>(hdr + kEpochWord) = e + 1u;
      *reinterpret_cast<volatile uint32_t*>(hdr + kStageDone) = 0u;
    }
  }
}

// Completion barrier over the windows' headers (no data): publish `epoch` into slot `rank` of every peer's header, then wait
// until every peer's slot in the LOCAL header has reached it.  Used after the fused render launch whose compositing epilogue
// stored this rank's row block of the frame straight into the root rank's window: when the root passes the barrier, every
// rank's stores have been performed at system scope (kernel boundary + fence.sys before the release store).
__global__ void peer_barrier_kernel(const Windows w, int world, int rank, uint32_t epoch, unsigned long long timeout_ns) {
  uint32_t* my_hdr = reinterpret_cast<uint32_t*>(w.base[rank]);
  int failed = 0;
  if (threadIdx.x < world) {
    __threadfence_system();
    st_release_sys(reinterpret_cast<uint32_t*>(w.base[threadIdx.x]) + kBarrierSlot0 + rank, epoch);
    if (threadIdx.x != rank) {
      const uint32_t* flag = my_hdr + kBarrierSlot0 + threadIdx.x;
      const unsigned long long t0 = global_ns();
      while ((int32_t)(ld_acquire_sys(flag) - epoch) < 0) {
        if (global_ns() - t0 > timeout_ns) {
          failed = 1;
          break;
        }
        __nanosleep(64);
      }
    }
  }
  failed = __syncthreads_or(failed);
  if (failed && threadIdx.x == 0) atomicMax(my_hdr + kStatusWord, epoch);
}

inline int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

// host array of `world` window pointers -> kernel argument; every window must be non-null and 256-byte aligned
inline int load_windows(void* const* windows, int world, Windows* w) {
  for (int p = 0; p < kMaxWorld; ++p) {
    w->base[p] = p < world ? static_cast<uint8_t*>(windows[p]) : nullptr;
    if (p < world && (w->base[p] == nullptr || (reinterpret_cast<uintptr_t>(w->base[p]) & 255u) != 0)) return TP_ERR_ALIGN;
  }
  return TP_OK;
}

}  // namespace

TP_API int64_t tp_peer_capacity_bytes(int64_t n_floats) { return n_floats < 0 ? 0 : round_up(n_floats * 4, 256); }

TP_API int64_t tp_peer_window_bytes(int64_t n_floats) {
  return n_floats < 0 ? 0 : kHeaderBytes + 2 * tp_peer_capacity_bytes(n_floats);
}

TP_API int64_t tp_peer_data_offset(int64_t n_floats, int parity) {
  return kHeaderBytes + (int64_t)(parity & 1) * tp_peer_capacity_bytes(n_floats);
}

TP_API int tp_peer_window_create(int64_t bytes, void** window_out) {
  if (bytes < kHeaderBytes || window_out == nullptr) return TP_ERR_BAD_ARG;
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, (size_t)bytes);
  if (e != cudaSuccess) return (int)e;
  e = cudaMemset(p, 0, (size_t)bytes);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    cudaFree(p);
    return (int)e;
  }
  *window_out = p;
  return TP_OK;
}

TP_API int tp_peer_window_destroy(void* window) {
  if (window == nullptr) return TP_OK;
  return (int)cudaFree(window);
}

TP_API int tp_peer_window_export(const void* window, void* handle64) {
  if (window == nullptr || handle64 == nullptr) return TP_ERR_BAD_ARG;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, const_cast<void*>(window));
  if (e != cudaSuccess) return (int)e;
  memcpy(handle64, &h, 64);
  return TP_OK;
}

TP_API int tp_peer_window_import(const void* handle64, void** window_out) {
  if (handle64 == nullptr || window_out == nullptr) return TP_ERR_BAD_ARG;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  void* p = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) return (int)e;
  *window_out = p;
  return TP_OK;
}

TP_API int tp_peer_window_release(void* imported_window) {
  if (imported_window == nullptr) return TP_OK;
  return (int)cudaIpcCloseMemHandle(imported_window);
}

TP_API int tp_peer_allreduce_mean(void* const* windows, int world, int rank, int64_t n_floats, uint32_t epoch, float* out,
                                  int grid_ctas, int64_t timeout_ms, void* stream) {
  if (windows == nullptr || out == nullptr || world < 1 || world > kMaxWorld || rank < 0 || rank >= world || n_floats < 0 ||
      epoch == 0)
    return TP_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(out) & 15u) != 0) return TP_ERR_ALIGN;
  Windows w;
  if (int rc = load_windows(windows, world, &w)) return rc;
  if (n_floats == 0) return TP_OK;
  const int64_t n4 = (n_floats + 3) / 4;   // buffers are padded to 256 B, `out` must hold round_up(n,4) floats
  int grid = grid_ctas > 0 ? grid_ctas : tp_grid_for(n4, 256, 2);
  if (timeout_ms <= 0) timeout_ms = 10000;
  peer_allreduce_mean_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      w, world, rank, n4, tp_peer_capacity_bytes(n_floats), epoch, out, (unsigned long long)timeout_ms * 1000000ull);
  return tp_launch_status();
}

TP_API int tp_peer_stage(void* window, int64_t n_floats, const float* src, void* stream) {
  if (window == nullptr || src == nullptr || n_floats < 0) return TP_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(window) & 255u) != 0 || (reinterpret_cast<uintptr_t>(src) & 15u) != 0) return TP_ERR_ALIGN;
  if (n_floats == 0) return TP_OK;
  peer_stage_kernel<<<tp_grid_for((n_floats + 3) / 4, 256, 2), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<uint8_t*>(window), n_floats, tp_peer_capacity_bytes(n_floats), src);
  return tp_launch_status();
}

TP_API int tp_peer_allreduce_mean_dev(void* const* windows, int world, int rank, int64_t n_floats, float* out, int grid_ctas,
                                      int64_t timeout_ms, void* stream) {
  if (windows == nullptr || out == nullptr || world < 1 || world > kMaxWorld || rank < 0 || rank >= world || n_floats < 0)
    return TP_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(out) & 15u) != 0) return TP_ERR_ALIGN;
  Windows w;
  if (int rc = load_windows(windows, world, &w)) return rc;
  if (n_floats == 0) return TP_OK;
  const int64_t n4 = (n_floats + 3) / 4;
  int grid = grid_ctas > 0 ? grid_ctas : tp_grid_for(n4, 256, 2);
  if (timeout_ms <= 0) timeout_ms = 10000;
  peer_allreduce_mean_dev_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      w, world, rank, n4, tp_peer_capacity_bytes(n_floats), out, (unsigned long long)timeout_ms * 1000000ull);
  return tp_launch_status();
}

TP_API int tp_peer_barrier(void* const* windows, int world, int rank, uint32_t epoch, int64_t timeout_ms, void* stream) {
  if (windows == nullptr || world < 1 || world > kMaxWorld || rank < 0 || rank >= world || epoch == 0) return TP_ERR_BAD_ARG;
  Windows w;
  if (int rc = load_windows(windows, world, &w)) return rc;
  if (timeout_ms <= 0) timeout_ms = 10000;
  peer_barrier_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(w, world, rank, epoch, (unsigned long long)timeout_ms * 1000000ull);
  return tp_launch_status();
}

TP_API int tp_peer_status(const void* window, uint32_t* status_host) {
  if (window == nullptr || status_host == nullptr) return TP_ERR_BAD_ARG;
  return (int)cudaMemcpy(status_host, static_cast<const uint8_t*>(window) + kStatusWord * 4, 4, cudaMemcpyDeviceToHost);
}
