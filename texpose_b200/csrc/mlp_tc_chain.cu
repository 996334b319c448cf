// K2b, staged variant: the dX chain of ANY stack of 256-wide ReLU layers on the tensor cores, stage list passed as data.
//
// mlp_tc_bwd.cu's fused chain is specialised for the two frozen-trunk heads of layers/nerf_static_transient_light.py.  The plain
// model (layers/nerf.py:61-99) trains its trunk as well, so its backward walks head + trunk: autograd of
//     h_l = relu(W_l h_{l-1} + b_l)      ->      dz_{l-1} = (dz_l W_l) * [h_{l-1} > 0]
// per 128-sample tile, with the ReLU bitmasks of the activations the single-pass forward saved (csrc/mlp_tc_split.cu) as masks and
// every dz tile stored as an image for the weight-gradient GEMMs (tp_tc_dw_gemm).  A stage may add one K = 16 step that reads a
// THIN operand (<= 8 fp32 columns per sample, turned into a bf16 tile by the drain warps): the gradient of a narrow output layer
// (dz_rgb: 3 columns) or of a single extra output row (the raw density, row 0 of the last trunk layer).
//
// Structure (one persistent 320-thread CTA per SM, one tile at a time): weights (transposed images, tp_tc_pack_weights) stream
// through a 4 x 16 KB ring, tcgen05.mma M = 128 x N = 256 into TWO 256-column TMEM accumulators used alternately by the stages,
// 8 drain warps mask / convert / write the next A operand in place -- published in eight 32-column groups, so the next stage's
// MMAs overlap the drain -- and stream the dz image to HBM from their registers.  The ReLU masks are the 4 KB bitmasks the forward
// wrote beside the tile images (a 64 KB mask tile per stage made the kernel HBM-bound at twice the traffic).  HBM per stage and
// tile: 4 KB of mask bits in + 64 KB dz out.
#include <cuda_bf16.h>
#include "tc_common.cuh"
#include "../../include/texpose_b200.h"

namespace tcc {
using namespace tc;

constexpr int kThreads = 320;        // warps 0-7 drain, warp 8 weight producer, warp 9 MMA issuer
constexpr int kRing = 4;
constexpr uint32_t kOffA = 0, kOffZ = kABytes;      // Z: two thin tiles [2 k8][128][8] (4 KB each)
constexpr uint32_t kOffRing = kOffZ + 8192;
constexpr uint32_t kOffBar = kOffRing + kRing * kChunkBytes;
constexpr uint32_t kSmemBytes = kOffBar + 256;
constexpr int kMaxStages = 16;

struct Stage {
  int thin, thin_chunk;      // thin >= 0: a K = 16 step on thin tile `thin` with the 8 KB chunk `thin_chunk` comes first
  int chunk0, n_chunks;      // then n_chunks (0 | 8) K = 32 chunks from `chunk0` on, read against the A tile
  int mask_slot, out_slot;   // saved activation whose positive entries pass (its ReLU bitmask); dz image slot written
};
struct Params {
  const float* thin[2];
  int thin_cols[2];
  long long S;
  const uint8_t* packed;     // transposed weight chunks (16 KB each)
  const uint32_t* bits;      // [tiles][n_saved][8 planes][128 rows] ReLU bitmasks of the saved activations
  int n_saved;
  uint8_t* dz_out;           // [tiles][n_out][64 KB]
  int n_out;
  int n_stages;
  Stage st[kMaxStages];
};

__global__ void __launch_bounds__(kThreads, 1) chain_backward_staged_kernel(const Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const uint32_t bar0 = sbase + kOffBar;
  auto bar_full = [&](int s) { return bar0 + 8 * s; };
  auto bar_empty = [&](int s) { return bar0 + 8 * (kRing + s); };
  // Both 256-column accumulators serve the one tile, alternating by stage, and the drain publishes the next A operand in eight
  // 32-column groups (= the eight K = 32 chunks of the next stage): the MMAs of stage s + 1 start after the first group and overlap
  // the rest of the drain of stage s (the mechanism of csrc/mlp_tc_split.cu; this kernel has no thin accumulators in its way).
  auto bar_acc = [&](int i) { return bar0 + 8 * (2 * kRing + i); };
  auto bar_ready = [&](int g) { return bar0 + 8 * (2 * kRing + 2 + g); };
  const uint32_t bar_thin = bar0 + 8 * (2 * kRing + 10);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffBar + 8 * (2 * kRing + 12));

  if (threadIdx.x == 0) {
    for (int s = 0; s < kRing; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_empty(s), 1);
    }
    mbar_init(bar_acc(0), 1);
    mbar_init(bar_acc(1), 1);
    for (int g = 0; g < 8; ++g) mbar_init(bar_ready(g), 4);      // the four lane-quarter warps of the column half
    mbar_init(bar_thin, 8);          // one arrive per drain warp: the tile's thin operands are in place, its last accumulator is read
    fence_barrier_init();
  }
  if (warp == 9) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const long long n_tiles = (p.S + 127) / 128;
  const int n_stages = p.n_stages;

  if (warp == 8) {
    // ================================================================ weight producer
    uint32_t slot = 0, phase = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      for (int s = 0; s < n_stages; ++s) {
        const Stage sg = p.st[s];
        const int n = (sg.thin >= 0 ? 1 : 0) + sg.n_chunks;
        for (int j = 0; j < n; ++j) {
          const bool thin = sg.thin >= 0 && j == 0;
          const int chunk = thin ? sg.thin_chunk : sg.chunk0 + j - (sg.thin >= 0 ? 1 : 0);
          const uint32_t bytes = thin ? kChunkBytes / 2 : kChunkBytes;
          mbar_wait(bar_empty(slot), phase ^ 1);
          if (elect_one_sync()) {
            mbar_expect_tx(bar_full(slot), bytes);
            bulk_g2s_hint(sbase + kOffRing + slot * kChunkBytes, p.packed + (size_t)chunk * kChunkBytes, bytes, bar_full(slot),
                          l2_policy_evict_last());
          }
          __syncwarp();
          if (++slot == kRing) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 9) {
    // ================================================================ MMA issuer
    uint32_t slot = 0, phase = 0, ready_ph = 0, thin_ph = 0, g = 0;
    const uint32_t idesc = umma_idesc(128, 256);
    constexpr uint32_t kHi = (128u >> 4) | (1u << 14);
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      mbar_wait(bar_thin, thin_ph);
      thin_ph ^= 1;
      for (int s = 0; s < n_stages; ++s, ++g) {
        const Stage sg = p.st[s];
        const int n = (sg.thin >= 0 ? 1 : 0) + sg.n_chunks;
        const uint32_t d_tmem = tmem_base + (g & 1u) * 256;
        for (int j = 0; j < n; ++j) {
          const bool thin = sg.thin >= 0 && j == 0;
          const int c = j - (sg.thin >= 0 ? 1 : 0);
          if (!thin) mbar_wait(bar_ready(c), ready_ph);      // columns [32 c, 32 c + 32) of the A tile are written
          mbar_wait(bar_full(slot), phase);
          tc_fence_after();
          if (elect_one_sync()) {
            const uint32_t wsm = sbase + kOffRing + slot * kChunkBytes;
            const uint32_t b_lo = (wsm >> 4) | ((4096u >> 4) << 16);
            if (thin) {
              const uint32_t a_lo = ((sbase + kOffZ + (uint32_t)sg.thin * 4096u) >> 4) | ((2048u >> 4) << 16);
              umma_bf16_lohi(d_tmem, a_lo, kHi, b_lo, kHi, idesc, 0u);
            } else {
              const uint32_t a_lo = ((sbase + kOffA + (uint32_t)c * 4u * 2048u) >> 4) | ((2048u >> 4) << 16);
              umma_bf16_lohi(d_tmem, a_lo, kHi, b_lo, kHi, idesc, j > 0 ? 1u : 0u);
              umma_bf16_lohi(d_tmem, a_lo + (4096u >> 4), kHi, b_lo + (8192u >> 4), kHi, idesc, 1u);
            }
            if (j == n - 1) umma_commit(bar_acc(g & 1u));
            umma_commit(bar_empty(slot));
          }
          __syncwarp();
          if (++slot == kRing) { slot = 0; phase ^= 1; }
        }
        if (sg.n_chunks) ready_ph ^= 1;
      }
    }
  } else {
    // ================================================================ drain warps: mask, convert, next A operand, dz image
    const int q = warp & 3, half = warp >> 2, row = q * 32 + lane;
    const uint32_t a_smem = sbase + kOffA;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16) + half * 128;
    uint32_t acc_ph = 0, g = 0;      // acc_ph bit i: phase of bar_acc(i)
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      // thin tiles of this tile's samples: [2 k8][128 rows][8] bf16, columns beyond the operand's width are zero
      if (half < 2 && p.thin[half]) {
        const long long s = tile * 128 + row;
        const int m = p.thin_cols[half];
        float z[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) z[c] = (s < p.S && c < m) ? p.thin[half][s * m + c] : 0.f;
        const uint32_t z0 = sbase + kOffZ + half * 4096 + row * 16;
        st_shared_v4(z0, pack_bf16(z[0], z[1]), pack_bf16(z[2], z[3]), pack_bf16(z[4], z[5]), pack_bf16(z[6], z[7]));
        st_shared_v4(z0 + 2048, 0u, 0u, 0u, 0u);
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_thin);

      for (int s = 0; s < n_stages; ++s, ++g) {
        const Stage sg = p.st[s];
        const bool last = s == n_stages - 1;
        // ReLU bitmask words of this thread's four 32-column slabs, fetched before the accumulator wait
        const uint32_t* bw = p.bits + ((size_t)tile * p.n_saved + sg.mask_slot) * 1024 + half * 4 * 128 + row;
        const uint32_t words[4] = {__ldg(bw), __ldg(bw + 128), __ldg(bw + 256), __ldg(bw + 384)};
        mbar_wait(bar_acc(g & 1u), (acc_ph >> (g & 1u)) & 1u);
        acc_ph ^= 1u << (g & 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_row + (g & 1u) * 256;
        uint8_t* g_tile = p.dz_out + ((size_t)tile * p.n_out + sg.out_slot) * kABytes;
        auto slab = [&](const uint32_t (&v)[32], int j) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint32_t off = (uint32_t)(half * 16 + j * 4 + i) * 2048 + row * 16;
            const uint32_t byte = (words[j] >> (i * 8)) & 0xffu;
            uint32_t o[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float lo = (byte & (1u << (2 * e))) ? __uint_as_float(v[i * 8 + 2 * e]) : 0.f;
              const float hi = (byte & (2u << (2 * e))) ? __uint_as_float(v[i * 8 + 2 * e + 1]) : 0.f;
              o[e] = pack_bf16(lo, hi);
            }
            st_shared_v4(a_smem + off, o[0], o[1], o[2], o[3]);
            st_global_cs_v4(g_tile + off, o[0], o[1], o[2], o[3]);
          }
          if (!last) {       // (the last stage's output feeds no MMA: its groups are not published)
            fence_proxy_async_smem();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_ready(half * 4 + j));
          }
        };
        uint32_t va[32], vb[32];
        TP_TMEM_LD32(tmem_d, va);
        TP_TMEM_WAIT32(va);
        TP_TMEM_LD32(tmem_d + 32, vb);
        slab(va, 0);
        TP_TMEM_WAIT32(vb);
        TP_TMEM_LD32(tmem_d + 64, va);
        slab(vb, 1);
        TP_TMEM_WAIT32(va);
        TP_TMEM_LD32(tmem_d + 96, vb);
        slab(va, 2);
        TP_TMEM_WAIT32(vb);
        slab(vb, 3);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// Column sums of tile images (bias gradients: db = sum over the samples of dz).  Block (x, y) walks the tiles x, x + gridDim.x, ...
// of the y-th selected slot; a warp owns four k8 groups, lane = row (512 contiguous bytes per load), 32 fp32 accumulators per
// thread over all its tiles, one warp reduction at the end -> partial[x][y][256].  Fixed order: deterministic.
__global__ void __launch_bounds__(256) images_colsum_kernel(const uint8_t* __restrict__ images, int n_slots, long long n_tiles,
                                                           const int* __restrict__ sel, float* __restrict__ partial) {
  const int slot = sel[blockIdx.y], warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float acc[4][8];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[i][e] = 0.f;
  for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const uint8_t* img = images + ((size_t)t * n_slots + slot) * kABytes;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint4 q = __ldcs(reinterpret_cast<const uint4*>(img + (warp * 4 + i) * 2048 + (j * 32 + lane) * 16));
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          acc[i][2 * e] += __uint_as_float(w[e] << 16);
          acc[i][2 * e + 1] += __uint_as_float(w[e] & 0xffff0000u);
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float v = acc[i][e];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) partial[((size_t)blockIdx.x * gridDim.y + blockIdx.y) * 256 + (warp * 4 + i) * 8 + e] = v;
    }
}


// ---------------------------------------------------------------------------------------------------------------------------
// K2c: the same dX chain in the fp32-parity mode.  Every operand is bf16 hi + lo (hi = bf16(x), lo = bf16(x - hi): ~16 significand
// bits with fp32's exponent range, so the 1e-6 .. 1e-9 gradients of a mean-normalised loss keep their bits, and scaling the loss by
// a power of two scales every result exactly), and every K = 16 step is three tcgen05.mma passes into the fp32 accumulator:
//        D += A_hi W_hi  +  A_hi W_lo  +  A_lo W_hi        (the dropped A_lo W_lo term is ~2^-17 relative)
// Weights stream as 16 KB K = 16 slots [W^T_hi 8 KB | W^T_lo 8 KB] (tp_tc_pack_weights_split), the geometry of the parity forward's
// ring.  The drain splits each masked dz into hi / lo, writes both A tiles and the images [tiles][2 n_out][64 KB] (slot 2k = hi,
// 2k + 1 = lo): the weight-gradient GEMMs and column-sum helpers read them as ordinary bf16 slots.  The masks are the bitmasks of
// the split-save forward, [tiles][n_saved][8 planes][128 rows], as in the single-pass chain.
// SMEM: A_hi 64K | A_lo 64K | Z_hi 8K | Z_lo 8K | ring 4 x 16K | barriers = 213 248 B.  TMEM: 512 columns.
namespace split {
constexpr uint32_t kOffAhi = 0, kOffAlo = kABytes, kOffZhi = 2 * kABytes, kOffZlo = kOffZhi + 8192;
constexpr uint32_t kOffRingS = kOffZlo + 8192;
constexpr uint32_t kOffBarS = kOffRingS + kRing * kChunkBytes;
constexpr uint32_t kSmemBytesS = kOffBarS + 256;
static_assert(kSmemBytesS <= 232448, "227 KB of shared memory per CTA");
constexpr int kStepsPerLayer = 16;      // K = 16 slots per 256-wide layer
}  // namespace split

__global__ void __launch_bounds__(kThreads, 1) chain_backward_split_kernel(const Params p) {
  using namespace split;
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const uint32_t bar0 = sbase + kOffBarS;
  auto bar_full = [&](int s) { return bar0 + 8 * s; };
  auto bar_empty = [&](int s) { return bar0 + 8 * (kRing + s); };
  auto bar_acc = [&](int i) { return bar0 + 8 * (2 * kRing + i); };
  auto bar_ready = [&](int g) { return bar0 + 8 * (2 * kRing + 2 + g); };      // 8: A columns [32g, 32g+32) written (hi and lo)
  const uint32_t bar_thin = bar0 + 8 * (2 * kRing + 10);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffBarS + 8 * (2 * kRing + 12));

  if (threadIdx.x == 0) {
    for (int s = 0; s < kRing; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_empty(s), 1);
    }
    mbar_init(bar_acc(0), 1);
    mbar_init(bar_acc(1), 1);
    for (int g = 0; g < 8; ++g) mbar_init(bar_ready(g), 4);
    mbar_init(bar_thin, 8);
    fence_barrier_init();
  }
  if (warp == 9) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const long long n_tiles = (p.S + 127) / 128;
  const int n_stages = p.n_stages;

  if (warp == 8) {
    // ================================================================ weight producer: one 16 KB slot per K = 16 step
    uint32_t slot = 0, phase = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      for (int s = 0; s < n_stages; ++s) {
        const Stage sg = p.st[s];
        const int n = (sg.thin >= 0 ? 1 : 0) + sg.n_chunks;
        for (int j = 0; j < n; ++j) {
          const int chunk = (sg.thin >= 0 && j == 0) ? sg.thin_chunk : sg.chunk0 + j - (sg.thin >= 0 ? 1 : 0);
          mbar_wait(bar_empty(slot), phase ^ 1);
          if (elect_one_sync()) {
            mbar_expect_tx(bar_full(slot), kChunkBytes);
            bulk_g2s_hint(sbase + kOffRingS + slot * kChunkBytes, p.packed + (size_t)chunk * kChunkBytes, kChunkBytes, bar_full(slot),
                          l2_policy_evict_last());
          }
          __syncwarp();
          if (++slot == kRing) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 9) {
    // ================================================================ MMA issuer: three passes per K = 16 step
    uint32_t slot = 0, phase = 0, ready_ph = 0, thin_ph = 0, g = 0;
    const uint32_t idesc = umma_idesc(128, 256);
    constexpr uint32_t kHi = (128u >> 4) | (1u << 14);
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      mbar_wait(bar_thin, thin_ph);
      thin_ph ^= 1;
      for (int s = 0; s < n_stages; ++s, ++g) {
        const Stage sg = p.st[s];
        const int n = (sg.thin >= 0 ? 1 : 0) + sg.n_chunks;
        const uint32_t d_tmem = tmem_base + (g & 1u) * 256;
        for (int j = 0; j < n; ++j) {
          const bool thin = sg.thin >= 0 && j == 0;
          const int ks = j - (sg.thin >= 0 ? 1 : 0);
          if (!thin && (ks & 1) == 0) mbar_wait(bar_ready(ks >> 1), ready_ph);      // columns [16 ks, 16 ks + 32) are written
          mbar_wait(bar_full(slot), phase);
          tc_fence_after();
          if (elect_one_sync()) {
            const uint32_t wsm = sbase + kOffRingS + slot * kChunkBytes;
            const uint32_t bh = (wsm >> 4) | ((4096u >> 4) << 16), bl = ((wsm + kChunkBytes / 2) >> 4) | ((4096u >> 4) << 16);
            const uint32_t a0 = thin ? kOffZhi + (uint32_t)sg.thin * 4096u : kOffAhi + (uint32_t)ks * 4096u;
            const uint32_t a1 = thin ? kOffZlo + (uint32_t)sg.thin * 4096u : kOffAlo + (uint32_t)ks * 4096u;
            const uint32_t ah = ((sbase + a0) >> 4) | ((2048u >> 4) << 16), al = ((sbase + a1) >> 4) | ((2048u >> 4) << 16);
            umma_bf16_lohi(d_tmem, ah, kHi, bh, kHi, idesc, j > 0 ? 1u : 0u);
            umma_bf16_lohi(d_tmem, ah, kHi, bl, kHi, idesc, 1u);
            umma_bf16_lohi(d_tmem, al, kHi, bh, kHi, idesc, 1u);
            if (j == n - 1) umma_commit(bar_acc(g & 1u));
            umma_commit(bar_empty(slot));
          }
          __syncwarp();
          if (++slot == kRing) { slot = 0; phase ^= 1; }
        }
        if (sg.n_chunks) ready_ph ^= 1;
      }
    }
  } else {
    // ================================================================ drain warps: mask, split, next A operand, dz images
    const int q = warp & 3, half = warp >> 2, row = q * 32 + lane;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16) + half * 128;
    uint32_t acc_ph = 0, g = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      // hi / lo thin tiles of this tile's samples: [2 k8][128 rows][8] bf16, columns beyond the operand's width are zero
      if (half < 2 && p.thin[half]) {
        const long long s = tile * 128 + row;
        const int m = p.thin_cols[half];
        float z[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) z[c] = (s < p.S && c < m) ? p.thin[half][s * m + c] : 0.f;
        uint32_t h[4], l[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) split2_bf16(z[2 * e], z[2 * e + 1], h[e], l[e]);
        const uint32_t z0 = sbase + kOffZhi + half * 4096 + row * 16, z1 = sbase + kOffZlo + half * 4096 + row * 16;
        st_shared_v4(z0, h[0], h[1], h[2], h[3]);
        st_shared_v4(z0 + 2048, 0u, 0u, 0u, 0u);
        st_shared_v4(z1, l[0], l[1], l[2], l[3]);
        st_shared_v4(z1 + 2048, 0u, 0u, 0u, 0u);
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_thin);

      for (int s = 0; s < n_stages; ++s, ++g) {
        const Stage sg = p.st[s];
        const bool last = s == n_stages - 1;
        const uint32_t* bw = p.bits + ((size_t)tile * p.n_saved + sg.mask_slot) * 1024 + half * 4 * 128 + row;
        const uint32_t words[4] = {__ldg(bw), __ldg(bw + 128), __ldg(bw + 256), __ldg(bw + 384)};
        mbar_wait(bar_acc(g & 1u), (acc_ph >> (g & 1u)) & 1u);
        acc_ph ^= 1u << (g & 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_row + (g & 1u) * 256;
        uint8_t* g_tile = p.dz_out + ((size_t)tile * 2 * p.n_out + 2 * sg.out_slot) * kABytes;      // hi; lo is the next slot
        auto slab = [&](const uint32_t (&v)[32], int j) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint32_t off = (uint32_t)(half * 16 + j * 4 + i) * 2048 + row * 16;
            const uint32_t byte = (words[j] >> (i * 8)) & 0xffu;
            uint32_t h[4], l[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float x0 = (byte & (1u << (2 * e))) ? __uint_as_float(v[i * 8 + 2 * e]) : 0.f;
              const float x1 = (byte & (2u << (2 * e))) ? __uint_as_float(v[i * 8 + 2 * e + 1]) : 0.f;
              split2_bf16(x0, x1, h[e], l[e]);
            }
            st_shared_v4(sbase + kOffAhi + off, h[0], h[1], h[2], h[3]);
            st_shared_v4(sbase + kOffAlo + off, l[0], l[1], l[2], l[3]);
            st_global_cs_v4(g_tile + off, h[0], h[1], h[2], h[3]);
            st_global_cs_v4(g_tile + kABytes + off, l[0], l[1], l[2], l[3]);
          }
          if (!last) {
            fence_proxy_async_smem();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_ready(half * 4 + j));
          }
        };
        uint32_t va[32], vb[32];
        TP_TMEM_LD32(tmem_d, va);
        TP_TMEM_WAIT32(va);
        TP_TMEM_LD32(tmem_d + 32, vb);
        slab(va, 0);
        TP_TMEM_WAIT32(vb);
        TP_TMEM_LD32(tmem_d + 64, va);
        slab(vb, 1);
        TP_TMEM_WAIT32(va);
        TP_TMEM_LD32(tmem_d + 96, vb);
        slab(va, 2);
        TP_TMEM_WAIT32(vb);
        slab(vb, 3);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// desc row as tp_tc_pack_weights' (10 int64: W ptr, ld, row0, rows_valid, col0, cols_valid, n_layout, bias ptr, bias k, transpose),
// with n_layout 256 and no bias: one K = 16 step (cols_valid <= 16) per 16 KB chunk, [2 k8][256 n][8] bf16 hi, then the same lo.
// transpose != 0: element (n, kl) = W[col0 + kl][row0 + n] (the B operand of dX = dZ W); else W[row0 + n][col0 + kl].
__global__ void pack_weights_split_kernel(const long long* __restrict__ desc, uint16_t* __restrict__ out) {
  const long long* d = desc + (long long)blockIdx.x * 10;
  const float* W = reinterpret_cast<const float*>(d[0]);
  const long long ld = d[1], row0 = d[2], rows_valid = d[3], col0 = d[4], cols_valid = d[5], transpose = d[9];
  uint16_t* o = out + (long long)blockIdx.x * (kChunkBytes / 2);
  for (int e = threadIdx.x; e < (int)(kChunkBytes / 4); e += blockDim.x) {
    const int kl = (e >> 11) * 8 + (e & 7), n = (e >> 3) & 255;
    float v = 0.f;
    if (W && n < rows_valid && kl < cols_valid) v = transpose ? W[(col0 + kl) * ld + row0 + n] : W[(row0 + n) * ld + col0 + kl];
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    o[e] = __bfloat16_as_ushort(hi);
    o[e + kChunkBytes / 4] = __bfloat16_as_ushort(__float2bfloat16_rn(v - __bfloat162float(hi)));
  }
}

}  // namespace tcc

TP_API int tp_tc_images_colsum_blocks(void) { return 32; }

/* out-of-place partials: partial [blocks][n_sel][256]; reduce with tp_reduce_partials(partial, blocks, n_sel * 256, out) */
TP_API int tp_tc_images_colsum(const void* images, int n_slots, int64_t S, const int32_t* sel, int n_sel, float* partial,
                               int64_t partial_floats, void* stream) {
  if (!images || !sel || !partial) return TP_ERR_BAD_ARG;
  if (n_slots < 1 || S < 1 || n_sel < 1 || n_sel > 64) return TP_ERR_BAD_SHAPE;
  const int blocks = tp_tc_images_colsum_blocks();
  if (partial_floats < (int64_t)blocks * n_sel * 256) return TP_ERR_WORKSPACE;
  tcc::images_colsum_kernel<<<dim3(blocks, n_sel), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint8_t*>(images), n_slots,
                                                                                  (S + 127) / 128, sel, partial);
  return tp_launch_status();
}

TP_API int tp_tc_chain_max_stages(void) { return tcc::kMaxStages; }

TP_API int tp_tc_chain_backward(const float* thin0, int cols0, const float* thin1, int cols1, int64_t S, const void* packed_bwd,
                                int n_chunks, const int32_t* stages, int n_stages, const void* mask_bits, int n_saved, void* dz_out,
                                int n_out, void* stream) {
  const void* saved = mask_bits;
  if (!thin0 || !packed_bwd || !stages || !saved || !dz_out) return TP_ERR_BAD_ARG;
  if (S < 0 || n_stages < 1 || n_stages > tcc::kMaxStages || n_saved < 1 || n_out < 1 || n_chunks < 1) return TP_ERR_BAD_SHAPE;
  if (cols0 < 1 || cols0 > 8 || (thin1 && (cols1 < 1 || cols1 > 8))) return TP_ERR_BAD_SHAPE;
  if (((uintptr_t)packed_bwd & 15) || ((uintptr_t)saved & 15) || ((uintptr_t)dz_out & 15)) return TP_ERR_ALIGN;
  if (!tp_device_is_sm100()) return TP_ERR_ARCH;
  tcc::Params p = {};
  for (int s = 0; s < n_stages; ++s) {
    const int32_t* r = stages + s * 6;
    tcc::Stage& sg = p.st[s];
    sg.thin = r[0]; sg.thin_chunk = r[1]; sg.chunk0 = r[2]; sg.n_chunks = r[3]; sg.mask_slot = r[4]; sg.out_slot = r[5];
    if (sg.thin < -1 || sg.thin > 1 || (sg.thin == 1 && !thin1)) return TP_ERR_BAD_ARG;
    if (sg.n_chunks != 0 && sg.n_chunks != 8) return TP_ERR_BAD_SHAPE;
    if (sg.thin < 0 && sg.n_chunks == 0) return TP_ERR_BAD_SHAPE;
    if (s == 0 && sg.n_chunks != 0) return TP_ERR_BAD_ARG;      // nothing has written the A tile yet
    if (s > 0 && sg.n_chunks == 0) return TP_ERR_BAD_ARG;       // every later stage consumes the previous drain's column groups
    if (sg.thin >= 0 && (sg.thin_chunk < 0 || sg.thin_chunk >= n_chunks)) return TP_ERR_BAD_ARG;
    if (sg.n_chunks && (sg.chunk0 < 0 || sg.chunk0 + sg.n_chunks > n_chunks)) return TP_ERR_BAD_ARG;
    if (sg.mask_slot < 0 || sg.mask_slot >= n_saved || sg.out_slot < 0 || sg.out_slot >= n_out) return TP_ERR_BAD_ARG;
  }
  if (S == 0) return TP_OK;
  p.thin[0] = thin0; p.thin[1] = thin1; p.thin_cols[0] = cols0; p.thin_cols[1] = thin1 ? cols1 : 0;
  p.S = S; p.packed = reinterpret_cast<const uint8_t*>(packed_bwd); p.bits = reinterpret_cast<const uint32_t*>(saved);
  p.n_saved = n_saved; p.dz_out = reinterpret_cast<uint8_t*>(dz_out); p.n_out = n_out; p.n_stages = n_stages;
  const long long n_tiles = (S + 127) / 128;
  int grid = tp_num_sms();
  if (n_tiles < grid) grid = (int)n_tiles;
  cudaError_t e = cudaFuncSetAttribute(tcc::chain_backward_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tcc::kSmemBytes);
  if (e != cudaSuccess) return (int)e;
  tcc::chain_backward_staged_kernel<<<grid, tcc::kThreads, tcc::kSmemBytes, (cudaStream_t)stream>>>(p);
  return tp_launch_status();
}

TP_API int tp_tc_pack_weights_split(const int64_t* chunk_desc, int n_chunks, void* packed, void* stream) {
  if (!chunk_desc || !packed) return TP_ERR_BAD_ARG;
  if (n_chunks < 1) return TP_ERR_BAD_SHAPE;
  if ((uintptr_t)packed & 15) return TP_ERR_ALIGN;
  tcc::pack_weights_split_kernel<<<n_chunks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const long long*>(chunk_desc),
                                                                          reinterpret_cast<uint16_t*>(packed));
  return tp_launch_status();
}

TP_API int tp_tc_chain_backward_split(const float* thin0, int cols0, const float* thin1, int cols1, int64_t S, const void* packed_bwd,
                                      int n_chunks, const int32_t* stages, int n_stages, const void* mask_bits, int n_saved,
                                      void* dz_out, int n_out, void* stream) {
  if (!thin0 || !packed_bwd || !stages || !mask_bits || !dz_out) return TP_ERR_BAD_ARG;
  if (S < 0 || n_stages < 1 || n_stages > tcc::kMaxStages || n_saved < 1 || n_out < 1 || n_chunks < 1) return TP_ERR_BAD_SHAPE;
  if (cols0 < 1 || cols0 > 8 || (thin1 && (cols1 < 1 || cols1 > 8))) return TP_ERR_BAD_SHAPE;
  if (((uintptr_t)packed_bwd & 15) || ((uintptr_t)mask_bits & 15) || ((uintptr_t)dz_out & 15)) return TP_ERR_ALIGN;
  tcc::Params p = {};
  for (int s = 0; s < n_stages; ++s) {
    const int32_t* r = stages + s * 6;
    tcc::Stage& sg = p.st[s];
    sg.thin = r[0]; sg.thin_chunk = r[1]; sg.chunk0 = r[2]; sg.n_chunks = r[3]; sg.mask_slot = r[4]; sg.out_slot = r[5];
    if (sg.thin < -1 || sg.thin > 1 || (sg.thin == 1 && !thin1)) return TP_ERR_BAD_ARG;
    if (sg.n_chunks != 0 && sg.n_chunks != tcc::split::kStepsPerLayer) return TP_ERR_BAD_SHAPE;
    if (sg.thin < 0 && sg.n_chunks == 0) return TP_ERR_BAD_SHAPE;
    if (s == 0 && sg.n_chunks != 0) return TP_ERR_BAD_ARG;      // nothing has written the A tiles yet
    if (s > 0 && sg.n_chunks == 0) return TP_ERR_BAD_ARG;       // every later stage consumes the previous drain's column groups
    if (sg.thin >= 0 && (sg.thin_chunk < 0 || sg.thin_chunk >= n_chunks)) return TP_ERR_BAD_ARG;
    if (sg.n_chunks && (sg.chunk0 < 0 || sg.chunk0 + sg.n_chunks > n_chunks)) return TP_ERR_BAD_ARG;
    if (sg.mask_slot < 0 || sg.mask_slot >= n_saved || sg.out_slot < 0 || sg.out_slot >= n_out) return TP_ERR_BAD_ARG;
  }
  if (!tp_device_is_sm100()) return TP_ERR_ARCH;
  if (S == 0) return TP_OK;
  p.thin[0] = thin0; p.thin[1] = thin1; p.thin_cols[0] = cols0; p.thin_cols[1] = thin1 ? cols1 : 0;
  p.S = S; p.packed = reinterpret_cast<const uint8_t*>(packed_bwd); p.bits = reinterpret_cast<const uint32_t*>(mask_bits);
  p.n_saved = n_saved; p.dz_out = reinterpret_cast<uint8_t*>(dz_out); p.n_out = n_out; p.n_stages = n_stages;
  const long long n_tiles = (S + 127) / 128;
  int grid = tp_num_sms();
  if (n_tiles < grid) grid = (int)n_tiles;
  cudaError_t e = cudaFuncSetAttribute(tcc::chain_backward_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)tcc::split::kSmemBytesS);
  if (e != cudaSuccess) return (int)e;
  tcc::chain_backward_split_kernel<<<grid, tcc::kThreads, tcc::split::kSmemBytesS, (cudaStream_t)stream>>>(p);
  return tp_launch_status();
}
