// Mask-prior frames (model/nerf_adapt_st_gan.py:633-680, render_by_slices for modes other than 'val'): the object-pixel ray list
// that the render launches take in list mode, and the defaults of the background pixels (:657-667) -- on the device, for B views,
// with no host read-back, so an eval frame is capturable in a CUDA graph.
//
// The list is built in three launches and without atomics (its order is fixed): per 4096-pixel chunk of a view the object count;
// one CTA scans the chunk counts of every view (padded view runs, view offsets, the total); per chunk a block scan places the
// chunk's pixels in ascending order.
#include "common.cuh"
#include "../../include/texpose_b200.h"

namespace tpmask {

constexpr int kThreads = 256, kPerThread = 16, kChunk = kThreads * kPerThread;

inline long long chunks_of(long long HW) { return (HW + kChunk - 1) / kChunk; }

// inclusive block scan of one value per thread (256 threads); `tmp` holds 8 warp totals
__device__ __forceinline__ long long block_scan(long long v, long long* tmp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long n = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += n;
  }
  if (lane == 31) tmp[warp] = v;
  __syncthreads();
  long long carry = 0;
  for (int w = 0; w < warp; ++w) carry += tmp[w];
  __syncthreads();
  return v + carry;
}

// this thread's pixels of chunk c of view b: [pix0, pix0 + n) (ascending), and how many of them are object pixels
__device__ __forceinline__ int thread_count(const float* __restrict__ mask, int b, long long c, long long HW, long long& pix0,
                                            int& n) {
  pix0 = c * kChunk + (long long)threadIdx.x * kPerThread;
  const long long left = HW - pix0;
  n = left <= 0 ? 0 : (left < kPerThread ? (int)left : kPerThread);
  const float* m = mask + (long long)b * HW + pix0;
  int k = 0;
  for (int i = 0; i < n; ++i) k += m[i] > 0.f;      // the reference's test: mask > 0 (NaN and -0 are background)
  return k;
}

// block (c, b): object pixels of chunk c of view b -> cnt[b * n_chunks + c]
__global__ void __launch_bounds__(kThreads) chunk_count_kernel(const float* __restrict__ mask, long long HW, long long* __restrict__ cnt) {
  __shared__ long long tmp[kThreads / 32];
  const long long c = blockIdx.x, n_chunks = gridDim.x;
  const int b = blockIdx.y;
  long long pix0;
  int n;
  const long long total = block_scan(thread_count(mask, b, c, HW, pix0, n), tmp);
  if (threadIdx.x == kThreads - 1) cnt[b * n_chunks + c] = total;
}

// one CTA: chunk counts -> chunk bases (exclusive, in list slots), per-view live counts, padded view starts, the total
__global__ void __launch_bounds__(kThreads) chunk_scan_kernel(long long* __restrict__ cnt, int B, long long n_chunks, int u,
                                                              long long* __restrict__ view0, int64_t* __restrict__ counts,
                                                              int64_t* __restrict__ n_slots) {
  __shared__ long long tmp[kThreads / 32], block_total;
  long long base = 0;      // first slot of the current view
  for (int b = 0; b < B; ++b) {
    long long carry = 0;   // object pixels of the view's earlier chunks
    for (long long c0 = 0; c0 < n_chunks; c0 += kThreads) {
      const long long c = c0 + threadIdx.x;
      const long long v = c < n_chunks ? cnt[b * n_chunks + c] : 0;
      const long long inc = block_scan(v, tmp);
      if (c < n_chunks) cnt[b * n_chunks + c] = base + carry + inc - v;
      if (threadIdx.x == kThreads - 1) block_total = inc;
      __syncthreads();
      carry += block_total;
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      counts[b] = carry;
      view0[b] = base;
    }
    base += (carry + u - 1) / u * u;
  }
  if (threadIdx.x == 0) *n_slots = base;
}

// block (c, b): the object pixels of chunk c of view b at their slots; the last chunk of a view also writes the view's pad entries
__global__ void __launch_bounds__(kThreads) chunk_place_kernel(const float* __restrict__ mask, long long HW, const long long* __restrict__ cnt,
                                                               const long long* __restrict__ view0, const int64_t* __restrict__ counts,
                                                               int u, int64_t* __restrict__ list) {
  __shared__ long long tmp[kThreads / 32];
  const long long c = blockIdx.x, n_chunks = gridDim.x;
  const int b = blockIdx.y;
  long long pix0;
  int n;
  const int k = thread_count(mask, b, c, HW, pix0, n);
  long long slot = cnt[b * n_chunks + c] + block_scan(k, tmp) - k;
  const float* m = mask + (long long)b * HW + pix0;
  for (int i = 0; i < n; ++i)
    if (m[i] > 0.f) list[slot++] = (long long)b * HW + pix0 + i;
  if (c == n_chunks - 1) {
    const long long live = counts[b], padded = (live + u - 1) / u * u;
    for (long long j = live + threadIdx.x; j < padded; j += kThreads) list[view0[b] + j] = ~((long long)b * HW);
  }
}

// Background defaults (:657-667) at pixels [pix0, pix1) of view blockIdx.y where mask <= 0: one thread per pixel and group of four
// samples (16-byte stores of the per-sample tensors; the pixel's per-ray defaults by its first group)
__global__ void defaults_kernel(const float* __restrict__ mask, long long HW, long long pix0, unsigned n_items, unsigned n4,
                                float min_uncert, float* rgb, float* rgb_s, float* rgb_t, float* depth, float* op, float* op_s,
                                float* op_t, float* unc, float4* as, float4* at, float4* density) {
  const long long b = blockIdx.y;
  const float4 one = make_float4(1.f, 1.f, 1.f, 1.f);
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += gridDim.x * blockDim.x) {
    const unsigned r = i / n4, k4 = i - r * n4;
    const long long q = b * HW + pix0 + r;      // frame position
    if (mask[q] > 0.f) continue;
    const long long s4 = q * n4 + k4;
    if (as) as[s4] = one;
    if (at) at[s4] = one;
    if (density) {
      density[2 * s4] = one;
      density[2 * s4 + 1] = one;
    }
    if (k4 == 0) {
      for (int ch = 0; ch < 3; ++ch) {
        if (rgb) rgb[q * 3 + ch] = 0.f;
        if (rgb_s) rgb_s[q * 3 + ch] = 0.f;
        if (rgb_t) rgb_t[q * 3 + ch] = 0.f;
      }
      if (depth) depth[q] = 0.f;
      if (op) op[q] = 0.f;
      if (op_s) op_s[q] = 0.f;
      if (op_t) op_t[q] = 0.f;
      if (unc) unc[q] = min_uncert;
    }
  }
}

}  // namespace tpmask

TP_API int64_t tp_mask_ray_list_capacity(int B, int64_t HW, int N) {
  if (B < 1 || HW < 1 || (N != 32 && N != 64 && N != 128)) return 0;
  const int64_t u = 256 / N;
  return (int64_t)B * ((HW + u - 1) / u * u);
}

TP_API int64_t tp_mask_ray_list_workspace(int B, int64_t HW) {
  if (B < 1 || HW < 1) return 0;
  return ((int64_t)B * tpmask::chunks_of(HW) + B) * 8;
}

TP_API int tp_mask_ray_list(const float* mask, int B, int64_t HW, int N, int64_t* list, int64_t list_cap, int64_t* n_slots,
                            int64_t* counts, void* workspace, int64_t ws_bytes, void* stream) {
  if (!mask || !list || !n_slots || !counts || !workspace) return TP_ERR_BAD_ARG;
  if (B < 1 || HW < 1 || B > 65535 || (N != 32 && N != 64 && N != 128)) return TP_ERR_BAD_SHAPE;
  if (list_cap < tp_mask_ray_list_capacity(B, HW, N)) return TP_ERR_BAD_SHAPE;
  if (ws_bytes < tp_mask_ray_list_workspace(B, HW)) return TP_ERR_WORKSPACE;
  if (((uintptr_t)workspace & 7) || ((uintptr_t)list & 7) || ((uintptr_t)n_slots & 7) || ((uintptr_t)counts & 7)) return TP_ERR_ALIGN;
  const long long n_chunks = tpmask::chunks_of(HW);
  if (n_chunks > 0x7fffffffLL) return TP_ERR_BAD_SHAPE;
  long long* cnt = reinterpret_cast<long long*>(workspace);
  long long* view0 = cnt + (long long)B * n_chunks;
  const int u = 256 / N;
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid((unsigned)n_chunks, (unsigned)B);
  tpmask::chunk_count_kernel<<<grid, tpmask::kThreads, 0, st>>>(mask, HW, cnt);
  tpmask::chunk_scan_kernel<<<1, tpmask::kThreads, 0, st>>>(cnt, B, n_chunks, u, view0, counts, n_slots);
  tpmask::chunk_place_kernel<<<grid, tpmask::kThreads, 0, st>>>(mask, HW, cnt, view0, counts, u, list);
  return tp_launch_status();
}

TP_API int tp_mask_defaults(const float* mask, int B, int64_t HW, int64_t pix0, int64_t pix1, int N, float min_uncert, float* rgb,
                            float* rgb_static, float* rgb_transient, float* depth, float* opacity, float* opacity_static,
                            float* opacity_transient, float* uncert, float* alpha_static, float* alpha_transient, float* density,
                            void* stream) {
  if (!mask) return TP_ERR_BAD_ARG;
  if (B < 1 || B > 65535 || HW < 1 || N < 4 || (N & 3) || pix0 < 0 || pix1 < pix0 || pix1 > HW) return TP_ERR_BAD_SHAPE;
  if (((uintptr_t)alpha_static & 15) || ((uintptr_t)alpha_transient & 15) || ((uintptr_t)density & 15)) return TP_ERR_ALIGN;
  const long long items = (pix1 - pix0) * (N / 4);      // per view
  if (items > 0x7fffffffLL) return TP_ERR_BAD_SHAPE;
  if (items == 0) return TP_OK;
  long long blocks = (items + 255) / 256;
  const long long cap = (long long)tp_num_sms() * 8;
  if (blocks * B > cap) blocks = (cap + B - 1) / B;
  tpmask::defaults_kernel<<<dim3((unsigned)blocks, (unsigned)B), 256, 0, (cudaStream_t)stream>>>(
      mask, HW, pix0, (unsigned)items, (unsigned)(N / 4), min_uncert, rgb, rgb_static, rgb_transient, depth, opacity, opacity_static,
      opacity_transient, uncert, reinterpret_cast<float4*>(alpha_static), reinterpret_cast<float4*>(alpha_transient),
      reinterpret_cast<float4*>(density));
  return tp_launch_status();
}
