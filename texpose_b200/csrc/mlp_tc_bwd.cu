// K2b (bf16 mode): tensor-core backward of the two NeRF heads (trunk frozen, layers/nerf_static_transient_light.py:34,87).
//
// autograd of the reference replays ~20 aten kernels per head layer; here the backward works on the bf16 *tile images*
// ([32 k8][128 rows][8], 64 KB per 128 samples) and ReLU bitmasks that the forward saved.  tp_tc_heads_backward (five launches,
// the yaml's 3 x 256 heads after the lock-step forward):
//
//   backward_chain_fused_kernel  dz3 -> dh3 = dz3 W3 -> dz2 = dh3*[h3>0] -> dh2 = dz2 W2 -> dz1 -> dh1 = dz1 W1 -> dz0 (per head)
//                                tcgen05 M=128 x N=256 MMAs, weights (transposed images) streamed like the forward, every dz
//                                tile stored as an image for the weight-gradient GEMMs; every thin gradient (biases, output
//                                layers, xyz / view columns, per-image sums) accumulated on the tensor pipe in the same kernel.
//   bwd_finish1/2_kernel         fixed-order reduction of the per-CTA thin partials, latent and layer-0 closed forms.
//   dw_gemm_kernel               dW[n,k] = sum_s dz[s,n] x[s,k]: both operands are read straight from the tile images as
//                                MN-major UMMA operands (the image of a [s x n] K-major tile IS the image of an [n x s] MN-major
//                                tile), full 256x256 fp32 accumulator in TMEM (2 x M=128), split over tiles across CTAs;
//                                dw_reduce_kernel reduces the splits in fixed order.
//
// dw_gemm_kernel and the HBM-bound helpers thin_dw / image_ray_sums / thin_colsum also serve the staged backward
// (csrc/mlp_tc_chain.cu, any 256-wide head depth, and batches whose images are too small for the fused chain kernel).
#include "tc_common.cuh"
#include "../../include/texpose_b200.h"

// cycle-counter instrumentation of the fused chain kernel (scripts/chain_prof.py): compiled in only with -DTP_CHAIN_PROF
#ifdef TP_CHAIN_PROF
#define TP_PF(...) __VA_ARGS__
#else
#define TP_PF(...)
#endif

namespace tcb {
using namespace tc;

constexpr int kThreads = 320;        // warps 0-7 epilogue, warp 8 weight producer, warp 9 MMA issuer
constexpr int kStages = 4;
constexpr uint32_t kOffA = 0;                        // dz operand tile (64 KB)
constexpr uint32_t kOffM = kABytes;                  // saved activation of the current stage (ReLU mask source, 64 KB)
constexpr uint32_t kOffZ = 2 * kABytes;              // dz3 tiles of the two heads: 2 x [2 k8][128][8] (4 KB each)
constexpr int kNumStagesPerTile = 6;                 // per head: output layer (K=16), hidden 2, hidden 1
constexpr int kBwdChunks = 34;                       // (1 + 8 + 8) x 2
constexpr int kFwdSlots = 7, kDzSlots = 6;
// forward-save slot holding the mask of each stage: rgb h3,h2,h1 = 3,2,1; trans h3,h2,h1 = 6,5,4
__constant__ int kMaskSlot[kNumStagesPerTile] = {3, 2, 1, 6, 5, 4};
// ReLU-bitmask slot (rgb h1, h2, trans h1, h2 = 0..3) that masks each stage of the fused kernel; -1: the h3 tile in M
__constant__ int kBitSlot[kNumStagesPerTile] = {-1, 1, 0, -1, 3, 2};

struct BwdParams {
  const float* dz_rgb;        // [S,3]  grad w.r.t. rgb-head output pre-activations
  const float* dz_trans;      // [S,5]
  long long S;
  const uint8_t* packed;      // kBwdChunks x 16 KB transposed weight images
  const uint8_t* saved;       // forward activations [tiles][7][64 KB]
  uint8_t* dz_out;            // [tiles][6][64 KB]: rgb dz2,dz1,dz0, trans dz2,dz1,dz0
};

// UMMA instruction descriptor with both operands MN-major (bits 15, 16)
__host__ __device__ constexpr uint32_t umma_idesc_mn(int M, int N) { return umma_idesc(M, N) | (1u << 15) | (1u << 16); }

// ------------------------------------------------------------------------------------------ fused chain + thin gradients
//
// The dX chain, plus every "thin" gradient of the two heads, computed by the otherwise idle tensor pipe while the operands are
// in SMEM anyway (the chain is HBM-bound).  All of them have the form  D[n, j] = sum_s X[s, n] * T[s, j]  with X a 128 x 256 tile
// image already resident (a dz tile in A, or the saved h3 tile in M) used as an MN-major A operand (2 x M=128 feature halves),
// and T a thin bf16 tile [128 samples x 16|48] built by the epilogue warps, used as an MN-major B operand:
//
//   block S  (N=16)  X = dz2 / dz1 of either head,   T = 1 in column {0,1,3,4}            -> bias gradients of layers 2, 1
//   block R  (N=48)  X = dz0 of the rgb head,        T = [image indicators 4 | xyz 3 | view encoding 27]
//                                                     -> per-image sums (bias, light-latent terms), dW columns of xyz / view
//   block T  (N=16)  X = dz0 of the transient head,  T = the same tile's first 16 columns  -> per-image sums (cols 0..3)
//   block O  (N=16)  X = h3 of a head (mask tile),   T = that head's dz3 tile              -> weight gradient of the output layer
//
// The accumulators (224 TMEM columns beside the chain's 256) run over ALL tiles of the CTA, which therefore processes a
// contiguous tile range; "image indicators" are relative to the first image the range touches (<= 4 images per CTA, checked by
// the host).  One flush per CTA at the end; bwd_finish_kernels reduce over CTAs in fixed order (deterministic).
constexpr uint32_t kOffTS = kOffZ + 8192;             // [2 k8][128][8]: a single 1-column, rewritten per stage
constexpr uint32_t kOffTI = kOffTS + 4096;            // 2 x [2 k8][128][8]: image-indicator tile (block T), by tile parity
constexpr uint32_t kOffTR = kOffTI + 2 * 4096;        // [6 k8][128][8]: indicator | xyz | view tile (block R)
constexpr uint32_t kTRBytes = 12288;
constexpr uint32_t kOffRingF = kOffTR + kTRBytes;
static_assert(kOffRingF + kStages * kChunkBytes + 128 <= 232448, "fused chain kernel exceeds 227 KB of shared memory");
constexpr uint32_t kOffBarF = kOffRingF + kStages * kChunkBytes;
constexpr uint32_t kSmemBytesF = kOffBarF + 128;
// TMEM columns of the extra accumulators (feature half h at +N*h)
constexpr uint32_t kColS = 256, kColT = 288, kColOr = 320, kColOt = 352, kColR = 384, kColRh = 64;
constexpr int kMaxImagesPerCta = 4;
// compact columns of the per-CTA partial [kXCols][256]
constexpr int kXdb = 0;        // 4: rgb db2, rgb db1, trans db2, trans db1
constexpr int kXimgR = 4;      // 4: per-image sums of rgb dz0 (local image index)
constexpr int kXxyz = 8;       // 3
constexpr int kXview = 11;     // 27
constexpr int kXimgT = 38;     // 4: per-image sums of trans dz0
constexpr int kXwr = 42;       // 3: rgb output-layer weight gradient rows
constexpr int kXwt = 45;       // 5: transient output-layer weight gradient rows
constexpr int kXCols = 50;

struct FusedParams {
  BwdParams b;
  const float* center;        // [rays,3]
  const float* ray;           // [rays,3]
  const float* depth;         // [S]
  int N;                      // samples per ray
  long long per_image;        // samples per image
  int L_view;
  float* extras;              // [grid][kXCols][256]
  float* thin_sums;           // [grid][4 warps][8]: column sums of dz_rgb (3) and dz_trans (5)
  long long* prof;            // optional [grid][16] cycle counters of the MMA warp and of epilogue warp 0 (debugging aid: workspace tail, see the API)
};

__device__ __forceinline__ void tile_range(long long n_tiles, int grid, int cta, long long& t0, long long& t1) {
  const long long per = n_tiles / grid, rem = n_tiles % grid;
  t0 = cta * per + (cta < rem ? cta : rem);
  t1 = t0 + per + (cta < rem ? 1 : 0);
}

// T_R row of one sample: [ind(4) | xyz(3) | u(3), per coord sin(2^k pi u) k<L, cos(...) k<L | 0...] as 48 bf16
__device__ __forceinline__ void write_tr_row(const FusedParams& p, long long s, long long img0, uint32_t dst_row,
                                             uint32_t ti_row) {
  float v[48];
#pragma unroll
  for (int i = 0; i < 48; ++i) v[i] = 0.f;
  if (s < p.b.S) {
    const long long r = s / p.N;
    const long long li = s / p.per_image - img0;
#pragma unroll
    for (int j = 0; j < kMaxImagesPerCta; ++j) v[j] = (li == j) ? 1.f : 0.f;
    const float d = p.depth[s];
    float dir[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      dir[j] = p.ray[r * 3 + j];
      v[4 + j] = __fadd_rn(p.center[r * 3 + j], __fmul_rn(dir[j], d));
    }
    const float len = fmaxf(sqrtf(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]), 1e-12f);
    const int L = p.L_view;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const float u = dir[j] / len;
      v[7 + j] = u;
      float sn, cs;
      sincospif(u, &sn, &cs);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (k < L) {
          v[10 + j * 2 * L + k] = sn;
          v[10 + j * 2 * L + L + k] = cs;
        }
        const float s2 = 2.f * sn * cs, c2 = (cs - sn) * (cs + sn);
        sn = s2;
        cs = c2;
      }
    }
  }
#pragma unroll
  for (int k8 = 0; k8 < 6; ++k8)
    st_shared_v4(dst_row + k8 * 2048, pack_bf16(v[k8 * 8], v[k8 * 8 + 1]), pack_bf16(v[k8 * 8 + 2], v[k8 * 8 + 3]),
                 pack_bf16(v[k8 * 8 + 4], v[k8 * 8 + 5]), pack_bf16(v[k8 * 8 + 6], v[k8 * 8 + 7]));
  st_shared_v4(ti_row, pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), 0u, 0u);
  st_shared_v4(ti_row + 2048, 0u, 0u, 0u, 0u);
}

constexpr int kFEpiWarps = 8, kFEpiThreads = kFEpiWarps * 32, kFThreads = kFEpiThreads + 64;   // + producer warp + MMA warp

__global__ void __launch_bounds__(kFThreads, 1) backward_chain_fused_kernel(const FusedParams fp) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const BwdParams& p = fp.b;
  const uint32_t sbase = smem_u32(smem);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const uint32_t bar0 = sbase + kOffBarF;
  auto bar_full = [&](int s) { return bar0 + 8 * s; };
  auto bar_empty = [&](int s) { return bar0 + 8 * (kStages + s); };
  const uint32_t bar_acc = bar0 + 8 * (2 * kStages), bar_ready = bar_acc + 8, bar_mask = bar_acc + 16;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffBarF + 8 * (2 * kStages + 3));

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_empty(s), 1);
    }
    mbar_init(bar_acc, 1);
    mbar_init(bar_ready, kFEpiWarps);      // one arrive per epilogue warp
    mbar_init(bar_mask, 1);
    fence_barrier_init();
  }
  if (warp == kFEpiWarps + 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const long long n_tiles = (p.S + 127) / 128;
  long long t0, t1;
  tile_range(n_tiles, gridDim.x, blockIdx.x, t0, t1);

  if (warp == kFEpiWarps) {
    // ================================================================ weight producer
    uint32_t stage = 0, phase = 0;
    for (long long tile = t0; tile < t1; ++tile) {
      int c = 0;
      for (int s = 0; s < kNumStagesPerTile; ++s) {
        const int nch = (s % 3 == 0) ? 1 : 8;
        for (int j = 0; j < nch; ++j, ++c) {
          const uint32_t bytes = (s % 3 == 0) ? kChunkBytes / 2 : kChunkBytes;
          mbar_wait(bar_empty(stage), phase ^ 1);
          if (elect_one_sync()) {
            mbar_expect_tx(bar_full(stage), bytes);
            bulk_g2s_hint(sbase + kOffRingF + stage * kChunkBytes, p.packed + (size_t)c * kChunkBytes, bytes, bar_full(stage), l2_policy_evict_last());
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kFEpiWarps + 1) {
    // ================================================================ MMA issuer: chain stages + thin-gradient MMAs
    uint32_t stage = 0, phase = 0, ready_ph = 0;
    const uint32_t idesc = umma_idesc(128, 256);
    const uint32_t idesc_x16 = umma_idesc_mn(128, 16), idesc_x48 = umma_idesc_mn(128, 48);
    constexpr uint32_t kHi = (128u >> 4) | (1u << 14);          // K-major operands: SBO 128
    constexpr uint32_t kHiMn = (2048u >> 4) | (1u << 14);       // MN-major operands: SBO 2048 (next 8 features / columns)
    const uint32_t a_tile = sbase + kOffA, m_tile = sbase + kOffM, ts_tile = sbase + kOffTS;
    // D[128 x n] (+)= X^T T over the 128 samples of the tile, for both feature halves
    auto thin_mma = [&](uint32_t col, uint32_t ncols, uint32_t x_tile, uint32_t t_tile, uint32_t id, bool first) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {
          const uint32_t a_lo = ((x_tile + h * 32768 + ks * 256) >> 4) | ((128u >> 4) << 16);
          const uint32_t b_lo = ((t_tile + ks * 256) >> 4) | ((128u >> 4) << 16);
          umma_bf16_lohi(tmem_base + col + h * ncols, a_lo, kHiMn, b_lo, kHiMn, id, (first && ks == 0) ? 0u : 1u);
        }
      }
    };
    TP_PF(long long pf_full = 0, pf_ready = 0, pf_mask = 0, pf_issue = 0;)
    TP_PF(const long long pf_t0 = clock64();)
    for (long long tile = t0; tile < t1; ++tile) {
      const uint32_t tr_tile = sbase + kOffTR;
      const uint32_t tr_prev = sbase + kOffTI + (uint32_t)((tile - t0 + 1) & 1) * 4096;
      const bool first_tile = tile == t0;
      for (int s = 0; s < kNumStagesPerTile; ++s) {
        const int nch = (s % 3 == 0) ? 1 : 8;
        for (int c = 0; c < nch; ++c) {
          TP_PF(long long pf_a = clock64();)
          mbar_wait(bar_full(stage), phase);
          TP_PF(long long pf_b = clock64();)
          TP_PF(pf_full += pf_b - pf_a;)
          if (c == 0) {
            mbar_wait(bar_ready, ready_ph);
            ready_ph ^= 1;
            TP_PF(pf_a = clock64();)
            TP_PF(pf_ready += pf_a - pf_b;)
            if (s % 3 == 0) mbar_wait(bar_mask, s == 3 ? 1u : 0u);        // h3 tile of this head (2 loads per tile): X operand of block O
            TP_PF(pf_b = clock64();)
            TP_PF(pf_mask += pf_b - pf_a;)
          }
          tc_fence_after();
          const uint32_t wsm = sbase + kOffRingF + stage * kChunkBytes;
          if (elect_one_sync()) {
            const uint32_t b_lo = (wsm >> 4) | ((4096u >> 4) << 16);
            if (s % 3 == 0) {   // K=16 step on the dz3 tile of this head
              const uint32_t a_lo = ((sbase + kOffZ + (s / 3) * 4096) >> 4) | ((2048u >> 4) << 16);
              umma_bf16_lohi(tmem_base, a_lo, kHi, b_lo, kHi, idesc, 0u);
            } else {
              const uint32_t a_lo = ((a_tile + c * 4 * 2048) >> 4) | ((2048u >> 4) << 16);
              umma_bf16_lohi(tmem_base, a_lo, kHi, b_lo, kHi, idesc, c > 0 ? 1u : 0u);
              umma_bf16_lohi(tmem_base, a_lo + (4096u >> 4), kHi, b_lo + (8192u >> 4), kHi, idesc, 1u);
            }
            if (c == (nch == 1 ? 0 : 1)) {
              // thin-gradient MMAs on the operands that are complete at this point; issued behind the first main MMAs so
              // their issue cost overlaps tensor-pipe work instead of delaying the stage (they only have to precede the
              // accumulator commit: the epilogue it releases overwrites A)
              if (s == 0) {
                if (tile > t0) thin_mma(kColT, 16, a_tile, tr_prev, idesc_x16, tile == t0 + 1);     // trans dz0 of the previous tile
                thin_mma(kColOr, 16, m_tile, sbase + kOffZ, idesc_x16, first_tile);
              } else if (s == 3) {
                thin_mma(kColR, kColRh, a_tile, tr_tile, idesc_x48, first_tile);                     // rgb dz0
                thin_mma(kColOt, 16, m_tile, sbase + kOffZ + 4096, idesc_x16, first_tile);
              } else {
                thin_mma(kColS, 16, a_tile, ts_tile, idesc_x16, first_tile && s == 1);              // dz2 / dz1 column sums
              }
            }
            if (c == nch - 1) umma_commit(bar_acc);
            umma_commit(bar_empty(stage));
          }
          __syncwarp();
          TP_PF(pf_issue += clock64() - pf_b;)
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    TP_PF(if (fp.prof && lane == 0) {
      long long* o = fp.prof + (size_t)blockIdx.x * 16;
      o[0] = clock64() - pf_t0; o[1] = pf_full; o[2] = pf_ready; o[3] = pf_mask; o[4] = pf_issue; o[5] = t1 - t0;
    })
    // trans dz0 of the last tile, then hand the accumulators to the flush
    mbar_wait(bar_ready, ready_ph);
    tc_fence_after();
    if (elect_one_sync()) {
      thin_mma(kColT, 16, a_tile, sbase + kOffTI + (uint32_t)((t1 - 1 - t0) & 1) * 4096, idesc_x16, t1 - t0 == 1);
      umma_commit(bar_acc);
    }
    __syncwarp();
  } else {
    // ================================================================ epilogue warps: mask, convert, store dz images, thin tiles
    // warp -> (TMEM lane quarter q, column half cq): each thread converts 128 accumulator columns (four 32-column slabs, the next
    // slab's TMEM load in flight while the current one is converted).  Eight drain warps, not sixteen: same-box A/B 2.218 vs 2.235 ms
    // per C3 step, and the narrower CTA leaves 168 registers per thread
    const int q = warp & 3, cq = warp >> 2, row = q * 32 + lane;
    const uint32_t a_smem = sbase + kOffA, m_smem = sbase + kOffM;
    const uint32_t tmem_d = tmem_base + ((uint32_t)(q * 32) << 16) + cq * 128;
    uint32_t acc_ph = 0, mask_ph = 0;
    const long long img0 = (t0 * 128) / fp.per_image;
    // ReLU bitmasks of h1 / h2 (written by the forward behind the tile images): word planes [8][128 rows] per tile and slot
    const uint8_t* bits = p.saved + ((p.S + 255) / 256) * 2 * (size_t)kFwdSlots * kABytes;
    float zsum[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    TP_PF(long long pe_acc = 0, pe_mask = 0, pe_store = 0, pe_conv = 0, pe_bar = 0;)
    if (threadIdx.x == 32) {
      mbar_expect_tx(bar_mask, kABytes);
      bulk_g2s_hint(m_smem, p.saved + ((size_t)t0 * kFwdSlots + kMaskSlot[0]) * kABytes, kABytes, bar_mask, l2_policy_evict_first());
    }
    // one 32-column slab: mask, bf16, store as 4 core-matrix rows of the dz tile (= next A operand / dz image)
    // ... and straight from the registers to the dz image in HBM (streaming 16-byte stores, a warp covers 512 contiguous bytes):
    // a 64 KB bulk store per stage would re-read the A tile through the shared-memory pipe the MMAs load, queue in the SM's TMA
    // FIFO in front of the next stage's weight chunks, and need a CTA barrier + wait before A may be overwritten
    auto convert_slab = [&](const uint32_t (&v)[32], int k8_0, bool tile_mask, uint32_t word, uint8_t* g_tile) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t off = (uint32_t)(k8_0 + i) * 2048 + row * 16;
        uint32_t o[4];
        if (tile_mask) {
          uint32_t m0, m1, m2, m3;
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(m0), "=r"(m1), "=r"(m2), "=r"(m3) : "r"(m_smem + off));
          const uint32_t mw[4] = {m0, m1, m2, m3};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float lo = (mw[e] & 0xffffu) ? __uint_as_float(v[i * 8 + 2 * e]) : 0.f;
            const float hi = (mw[e] >> 16) ? __uint_as_float(v[i * 8 + 2 * e + 1]) : 0.f;
            o[e] = pack_bf16(lo, hi);
          }
        } else {
          const uint32_t byte = (word >> (i * 8)) & 0xffu;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float lo = (byte & (1u << (2 * e))) ? __uint_as_float(v[i * 8 + 2 * e]) : 0.f;
            const float hi = (byte & (2u << (2 * e))) ? __uint_as_float(v[i * 8 + 2 * e + 1]) : 0.f;
            o[e] = pack_bf16(lo, hi);
          }
        }
        st_shared_v4(a_smem + off, o[0], o[1], o[2], o[3]);
        st_global_cs_v4(g_tile + off, o[0], o[1], o[2], o[3]);
      }
    };
    for (long long tile = t0; tile < t1; ++tile) {
      const long long s_row = tile * 128 + row;
      if (cq == 0) {
        // dz3 tiles of both heads: [2 k8][128 rows][8] bf16, columns >= 3 / 5 zero
        float zr[3] = {0.f, 0.f, 0.f}, zt[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        if (s_row < p.S) {
#pragma unroll
          for (int c = 0; c < 3; ++c) zr[c] = p.dz_rgb[s_row * 3 + c];
#pragma unroll
          for (int c = 0; c < 5; ++c) zt[c] = p.dz_trans[s_row * 5 + c];
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) zsum[c] += zr[c];
#pragma unroll
        for (int c = 0; c < 5; ++c) zsum[3 + c] += zt[c];
        const uint32_t z0 = sbase + kOffZ + row * 16;
        st_shared_v4(z0, pack_bf16(zr[0], zr[1]), pack_bf16(zr[2], 0.f), 0u, 0u);
        st_shared_v4(z0 + 2048, 0u, 0u, 0u, 0u);
        st_shared_v4(z0 + 4096, pack_bf16(zt[0], zt[1]), pack_bf16(zt[2], zt[3]), pack_bf16(zt[4], 0.f), 0u);
        st_shared_v4(z0 + 4096 + 2048, 0u, 0u, 0u, 0u);
      } else if (cq == 1) {
        write_tr_row(fp, s_row, img0, sbase + kOffTR + row * 16, sbase + kOffTI + (uint32_t)((tile - t0) & 1) * 4096 + row * 16);
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();                 // every lane's st.shared + proxy fence precede the warp's single arrive
      if (lane == 0) mbar_arrive(bar_ready);

      for (int s = 0; s < kNumStagesPerTile; ++s) {
        const bool tile_mask = s % 3 == 0;       // stages 0 / 3 mask with the h3 tile in M (it is also block O's operand)
        uint32_t w0 = 0u, w1 = 0u, w2 = 0u, w3 = 0u;
        if (!tile_mask) {                        // others: h2 / h1 bitmask words of this thread's 128 columns, fetched before the wait
          const uint32_t* w = reinterpret_cast<const uint32_t*>(bits + ((size_t)tile * 4 + kBitSlot[s]) * 4096) + cq * 4 * 128 + row;
          w0 = __ldg(w);
          w1 = __ldg(w + 128);
          w2 = __ldg(w + 256);
          w3 = __ldg(w + 384);
        }
        TP_PF(long long pe_a = clock64();)
        mbar_wait(bar_acc, acc_ph);
        acc_ph ^= 1;
        TP_PF(long long pe_b = clock64();)
        TP_PF(pe_acc += pe_b - pe_a;)
        if (tile_mask) {
          mbar_wait(bar_mask, mask_ph);
          mask_ph ^= 1;
        }
        tc_fence_after();
        TP_PF(pe_a = clock64();)
        TP_PF(pe_mask += pe_a - pe_b;)
        // (10 warps: up to 168 registers per thread -- the next slab's TMEM load is in flight while the current one is converted)
        uint32_t va[32], vb[32];
        TP_TMEM_LD32(tmem_d, va);
        uint8_t* g_tile = p.dz_out + ((size_t)tile * kDzSlots + s) * kABytes;
        TP_PF(pe_b = clock64();)
        TP_PF(pe_store += pe_b - pe_a;)
        TP_TMEM_WAIT32(va);
        TP_TMEM_LD32(tmem_d + 32, vb);
        convert_slab(va, cq * 16, tile_mask, w0, g_tile);
        TP_TMEM_WAIT32(vb);
        TP_TMEM_LD32(tmem_d + 64, va);
        convert_slab(vb, cq * 16 + 4, tile_mask, w1, g_tile);
        TP_TMEM_WAIT32(va);
        TP_TMEM_LD32(tmem_d + 96, vb);
        convert_slab(va, cq * 16 + 8, tile_mask, w2, g_tile);
        TP_TMEM_WAIT32(vb);
        convert_slab(vb, cq * 16 + 12, tile_mask, w3, g_tile);
        if (cq == 1 && s % 3 != 2) {       // the 1-column of block S for the dz tile just written: column = dz slot
          const uint32_t one = 0x3F80u << ((s & 1) * 16);
          const int w = s >> 1;
          st_shared_v4(sbase + kOffTS + row * 16, w == 0 ? one : 0u, w == 1 ? one : 0u, w == 2 ? one : 0u, 0u);
          st_shared_v4(sbase + kOffTS + 2048 + row * 16, 0u, 0u, 0u, 0u);
        }
        fence_proxy_async_smem();
        TP_PF(pe_a = clock64();)
        TP_PF(pe_conv += pe_a - pe_b;)
        if (tile_mask) named_bar_sync(1, kFEpiThreads);  // every thread finished reading M (the next h3 tile may land in it)
        TP_PF(pe_bar += clock64() - pe_a;)
        if (threadIdx.x == 32 && tile_mask) {    // M is free again: fetch the next h3 tile (trans h3 of this tile / rgb h3 of the next)
          const long long nt = s == 3 ? tile + 1 : tile;
          if (nt < t1) {
            mbar_expect_tx(bar_mask, kABytes);
            bulk_g2s_hint(m_smem, p.saved + ((size_t)nt * kFwdSlots + kMaskSlot[s == 3 ? 0 : 3]) * kABytes, kABytes, bar_mask, l2_policy_evict_first());
          }
        }
        if (s != kNumStagesPerTile - 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_ready);
        }
      }
    }
    // last tile: release the trans-dz0 thin MMA, then flush the thin accumulators of this CTA
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_ready);
    mbar_wait(bar_acc, acc_ph);
    tc_fence_after();
    if (cq < 2) {                                 // column halves 0 / 1 flush the accumulators of feature half 0 / 1
      const int half = cq, n = half * 128 + row;
      float* P = fp.extras + (size_t)blockIdx.x * kXCols * 256 + n;
      const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
      auto flush = [&](uint32_t col, int ncols, int x0, int src0) {   // TMEM columns [col, col+8) -> P[x0 + i] for i < ncols (from src0)
        uint32_t v[8];
        TP_TMEM_LD8(lane_addr + col, v);
        TP_TMEM_WAIT8(v);
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (i >= src0 && i < src0 + ncols) P[(size_t)(x0 + i - src0) * 256] = __uint_as_float(v[i]);
      };
      const uint32_t cS = kColS + half * 16, cT = kColT + half * 16, cOr = kColOr + half * 16, cOt = kColOt + half * 16;
      const uint32_t cR = kColR + half * kColRh;
      flush(cS, 2, kXdb, 0);            // slots 0, 1
      flush(cS, 2, kXdb + 2, 3);        // slots 3, 4
      flush(cR, 4, kXimgR, 0);
      flush(cR, 3, kXxyz, 4);
      flush(cR, 1, kXview, 7);
      flush(cR + 8, 8, kXview + 1, 0);
      flush(cR + 16, 8, kXview + 9, 0);
      flush(cR + 24, 8, kXview + 17, 0);
      flush(cR + 32, 2, kXview + 25, 0);
      flush(cT, 4, kXimgT, 0);
      flush(cOr, 3, kXwr, 0);
      flush(cOt, 5, kXwt, 0);
    }
    if (cq == 0) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float v = zsum[c];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) fp.thin_sums[((size_t)blockIdx.x * 4 + q) * 8 + c] = v;
      }
    }
    if (threadIdx.x == 0) bulk_wait_all();
    TP_PF(if (fp.prof && threadIdx.x == 0) {
      long long* o = fp.prof + (size_t)blockIdx.x * 16 + 8;
      o[0] = pe_acc; o[1] = pe_mask; o[2] = pe_store; o[3] = pe_conv; o[4] = pe_bar;
    })
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kFEpiWarps + 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ------------------------------------------------------------------------------------------ dW = dz^T x on tile images

constexpr uint32_t kDwSlots = 3;                     // ring of 64 KB image slots: A_i, B_i, A_{i+1}, ...
constexpr uint32_t kDwOffBar = kDwSlots * kABytes;
constexpr uint32_t kDwSmemBytes = kDwOffBar + 128;

constexpr int kDwMaxJobs = 12;      // (six head layers of the frozen-trunk model; up to 8 + the encoding jobs of the plain model)
struct DwParams {
  const uint8_t* a_images; int a_nslots;             // dz  (M = n)
  const uint8_t* b_images; int b_nslots;             // x   (N = k)
  int a_slot[kDwMaxJobs], b_slot[kDwMaxJobs];        // job j: dW_j = dz[a_slot[j]]^T x[b_slot[j]]
  int n_jobs, splits;                                // CTA -> (job = blockIdx % n_jobs, split = blockIdx / n_jobs)
  long long n_tiles;
  float* partial;                                    // [splits][n_jobs][256][256]
};


__global__ void __launch_bounds__(kThreads, 1) dw_gemm_kernel(const DwParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const uint32_t bar0 = sbase + kDwOffBar;
  auto bar_full = [&](int s) { return bar0 + 8 * s; };
  auto bar_empty = [&](int s) { return bar0 + 8 * (kDwSlots + s); };
  const uint32_t bar_acc = bar0 + 8 * (2 * kDwSlots);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kDwOffBar + 8 * (2 * kDwSlots + 1));
  if (threadIdx.x == 0) {
    for (int s = 0; s < (int)kDwSlots; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_empty(s), 1);
    }
    mbar_init(bar_acc, 1);
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
  // job and contiguous tile range of this CTA
  const int job = blockIdx.x % p.n_jobs, split = blockIdx.x / p.n_jobs;
  const long long per = p.n_tiles / p.splits, rem = p.n_tiles % p.splits;
  const long long t0 = split * per + (split < rem ? split : rem);
  const long long t1 = t0 + per + (split < rem ? 1 : 0);
  const int a_slot = p.a_slot[job], b_slot = p.b_slot[job];

  if (warp == 8) {
    uint32_t slot = 0, phase = 0;
    for (long long t = t0; t < t1; ++t) {
      for (int op = 0; op < 2; ++op) {
        const uint8_t* src = op == 0 ? p.a_images + ((size_t)t * p.a_nslots + a_slot) * kABytes
                                     : p.b_images + ((size_t)t * p.b_nslots + b_slot) * kABytes;
        mbar_wait(bar_empty(slot), phase ^ 1);
        if (elect_one_sync()) {
          mbar_expect_tx(bar_full(slot), kABytes);
          bulk_g2s(sbase + slot * kABytes, src, kABytes, bar_full(slot));
        }
        __syncwarp();
        if (++slot == kDwSlots) { slot = 0; phase ^= 1; }
      }
    }
  } else if (warp == 9) {
    uint32_t slot = 0, phase = 0;
    const uint32_t idesc = umma_idesc_mn(128, 256);
    // MN-major canonical layout of a tile image: 8 (K=s) x 8 (MN) core matrices, K-block stride (LBO) 128 B,
    // MN-block stride (SBO) 2048 B
    constexpr uint32_t lbo = 128u, sbo = 2048u;
    const uint32_t hi = (sbo >> 4) | (1u << 14);
    for (long long t = t0; t < t1; ++t) {
      const uint32_t sa = slot, pa = phase;
      if (++slot == kDwSlots) { slot = 0; phase ^= 1; }
      const uint32_t sb = slot, pb = phase;
      if (++slot == kDwSlots) { slot = 0; phase ^= 1; }
      mbar_wait(bar_full(sa), pa);
      mbar_wait(bar_full(sb), pb);
      tc_fence_after();
      if (elect_one_sync()) {
        const uint32_t a_base = sbase + sa * kABytes, b_base = sbase + sb * kABytes;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {
            const uint32_t a_lo = ((a_base + h * 32768 + ks * 256) >> 4) | ((lbo >> 4) << 16);
            const uint32_t b_lo = ((b_base + ks * 256) >> 4) | ((lbo >> 4) << 16);
            umma_bf16_lohi(tmem_base + h * 256, a_lo, hi, b_lo, hi, idesc, (t > t0 || ks > 0) ? 1u : 0u);
          }
        }
        umma_commit(bar_empty(sa));
        umma_commit(bar_empty(sb));
        if (t == t1 - 1) umma_commit(bar_acc);
      }
      __syncwarp();
    }
  } else {
    // epilogue: accumulator rows n (TMEM lanes) x columns k -> partial[cta][n][k]
    const int q = warp & 3, h = warp >> 2, n = h * 128 + q * 32 + lane;
    float* out = p.partial + (((size_t)split * p.n_jobs + job) * 256 + n) * 256;
    if (t1 > t0) {
      mbar_wait(bar_acc, 0);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + ((uint32_t)(q * 32) << 16) + h * 256;
#pragma unroll 1
      for (int j = 0; j < 8; ++j) {
        uint32_t v[32];
        TP_TMEM_LD32(tmem_d + j * 32, v);
        TP_TMEM_WAIT32(v);
#pragma unroll
        for (int i = 0; i < 32; i += 4)
          *reinterpret_cast<float4*>(out + j * 32 + i) = make_float4(__uint_as_float(v[i]), __uint_as_float(v[i + 1]),
                                                                     __uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
      }
    } else {
      for (int k = 0; k < 256; k += 4) *reinterpret_cast<float4*>(out + k) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ------------------------------------------------------------------------------------------ finish: per-CTA partials -> gradients

struct FinishParams {
  const float* extras;        // [grid][kXCols][256]
  const float* thin_sums;     // [grid][4][8]
  int grid;
  long long n_tiles, per_image;
  int B, vc, n_light, n_trans;
  float* tot;                 // [kXCols][256] column totals over the CTAs (indicator columns unused)
  float* img;                 // [2][4][B][256] per-image sums of rgb dz0 / transient dz0, one slab per indicator column
  const float* W_r0; long long ld_r0;      // mlp_rgb[0].weight  [256, 256 + vc + 3 + n_light]
  const float* W_t0; long long ld_t0;      // mlp_trans[0].weight [256, 256 + n_trans]
  const float* lat_light;     // [B, n_light]
  const float* lat_trans;     // [B, n_trans]
  float* g[16];               // rgb {dW0, db0, dW1, db1, dW2, db2, dW3, db3}, transient likewise (dW1, dW2 come from the GEMM)
  float* d_lat_light;         // [B, n_light] or NULL
  float* d_lat_trans;         // [B, n_trans] or NULL
};

// one block per compact column; fixed CTA order.  Indicator columns: column j of a CTA holds the sum over the samples of
// image (first image of the CTA's range + j) -> segmented sum over the CTAs into imgj[head][j][b][:] (images a (CTA, j) pair
// never touches stay zero; finish2 adds the four j slabs).
__global__ void __launch_bounds__(256) bwd_finish1_kernel(const FinishParams f) {
  __shared__ int img0_s[1024];
  const int c = blockIdx.x, n = threadIdx.x;
  const bool ind_r = c >= kXimgR && c < kXimgR + kMaxImagesPerCta, ind_t = c >= kXimgT && c < kXimgT + kMaxImagesPerCta;
  const float* src = f.extras + (size_t)c * 256 + n;
  const size_t stride = (size_t)kXCols * 256;
  if (!ind_r && !ind_t) {
    float acc = 0.f;
    int cta = 0;
    for (; cta + 8 <= f.grid; cta += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = src[(size_t)(cta + u) * stride];
#pragma unroll
      for (int u = 0; u < 8; ++u) acc += v[u];
    }
    for (; cta < f.grid; ++cta) acc += src[(size_t)cta * stride];
    f.tot[c * 256 + n] = acc;
    return;
  }
  for (int cta = n; cta < f.grid; cta += 256) {
    long long t0, t1;
    tile_range(f.n_tiles, f.grid, cta, t0, t1);
    img0_s[cta] = (int)((t0 * 128) / f.per_image);
  }
  __syncthreads();
  const int j = ind_r ? c - kXimgR : c - kXimgT;
  float* out = f.img + ((size_t)(ind_t ? 1 : 0) * kMaxImagesPerCta + j) * f.B * 256 + n;
  for (int b = 0; b < f.B; ++b) out[(size_t)b * 256] = 0.f;
  int cur = -1;
  float acc = 0.f;
  for (int cta0 = 0; cta0 < f.grid; cta0 += 8) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = cta0 + u < f.grid ? src[(size_t)(cta0 + u) * stride] : 0.f;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      if (cta0 + u >= f.grid) break;
      const int b = img0_s[cta0 + u] + j;
      if (b != cur) {
        if (cur >= 0 && cur < f.B) out[(size_t)cur * 256] = acc;
        cur = b;
        acc = 0.f;
      }
      acc += v[u];
    }
  }
  if (cur >= 0 && cur < f.B) out[(size_t)cur * 256] = acc;
}

constexpr int kFinishParts = 8;      // 8 latent columns each (n_latent <= 64)
// blocks 0..B-1: latent gradients of image b; then kFinishParts blocks per head for the thin outputs of that head
__global__ void __launch_bounds__(256) bwd_finish2_kernel(const FinishParams f) {
  const int n = threadIdx.x;
  extern __shared__ float gsm[];       // blocks < B: [2][256] sums of image b; blocks >= B: nothing
  const size_t slab = (size_t)f.B * 256;
  auto image_sum = [&](int head, int b, int i) {
    const float* q = f.img + (size_t)head * kMaxImagesPerCta * slab + (size_t)b * 256 + i;
    return ((q[0] + q[slab]) + q[2 * slab]) + q[3 * slab];
  };
  if ((int)blockIdx.x < f.B) {
    const int b = blockIdx.x;
    gsm[n] = image_sum(0, b, n);
    gsm[256 + n] = image_sum(1, b, n);
    __syncthreads();
    if (n < f.n_light && f.d_lat_light) {
      float acc = 0.f;
      for (int i = 0; i < 256; ++i) acc = fmaf(gsm[i], f.W_r0[i * f.ld_r0 + 256 + f.vc + 3 + n], acc);
      f.d_lat_light[b * f.n_light + n] = acc;
    } else if (n >= 64 && n - 64 < f.n_trans && f.d_lat_trans) {
      const int k = n - 64;
      float acc = 0.f;
      for (int i = 0; i < 256; ++i) acc = fmaf(gsm[256 + i], f.W_t0[i * f.ld_t0 + 256 + k], acc);
      f.d_lat_trans[b * f.n_trans + k] = acc;
    }
    return;
  }
  // blocks B .. B + 2 * kFinishParts - 1: (head, part); a part owns 8 latent columns of layer 0, part 0 also the rest
  const int hb = (int)blockIdx.x - f.B, head = hb / kFinishParts, part = hb % kFinishParts;
  const bool trans = head == 1;
  float* const* g = f.g + (trans ? 8 : 0);
  const int n_lat = trans ? f.n_trans : f.n_light;
  const float* lat = trans ? f.lat_trans : f.lat_light;
  const long long ld = trans ? f.ld_t0 : f.ld_r0;
  float* row = g[0] + (size_t)n * ld + 256 + (trans ? 0 : f.vc + 3);
  const int k0 = part * 8;
  if (k0 < n_lat) {
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int b = 0; b < f.B; ++b) {
      const float gb = image_sum(head, b, n);
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (k0 + k < n_lat) acc[k] = fmaf(gb, lat[b * n_lat + k0 + k], acc[k]);
    }
#pragma unroll
    for (int k = 0; k < 8; ++k)
      if (k0 + k < n_lat) row[k0 + k] = acc[k];
  }
  if (part != 0) return;
  g[5][n] = f.tot[(kXdb + (trans ? 2 : 0)) * 256 + n];          // db2
  g[3][n] = f.tot[(kXdb + (trans ? 3 : 1)) * 256 + n];          // db1
  float b0 = 0.f;
  for (int b = 0; b < f.B; ++b) b0 += image_sum(head, b, n);
  g[1][n] = b0;                                                  // db0
  if (!trans) {
    float* vrow = g[0] + (size_t)n * f.ld_r0 + 256;
    for (int i = 0; i < f.vc; ++i) vrow[i] = f.tot[(kXview + i) * 256 + n];
    for (int j = 0; j < 3; ++j) vrow[f.vc + j] = f.tot[(kXxyz + j) * 256 + n];
    for (int j = 0; j < 3; ++j) g[6][j * 256 + n] = f.tot[(kXwr + j) * 256 + n];
  } else {
    for (int j = 0; j < 5; ++j) g[6][j * 256 + n] = f.tot[(kXwt + j) * 256 + n];
  }
  // db3: warp j sums column j of the per-warp partials -- every lane a contiguous block in order, lane 0 the 32 block sums in
  // order (fixed order, 19 instead of 592 dependent loads)
  const int nb = trans ? 5 : 3, off = trans ? 3 : 0;
  const int wj = n >> 5, ln = n & 31;
  if (wj < nb) {
    const int items = f.grid * 4, per = (items + 31) / 32;
    float acc = 0.f;
    for (int i = ln * per; i < (ln + 1) * per && i < items; ++i) acc += f.thin_sums[(size_t)i * 8 + off + wj];
    float tot = 0.f;
    for (int l = 0; l < 32; ++l) tot += __shfl_sync(0xffffffffu, acc, l);
    if (ln == 0) g[7][wj] = tot;                                 // db3
  }
}

// second stage of the weight-gradient GEMMs, writing each job with its own leading dimension (no torch.cat afterwards)
struct DwOut { float* ptr[kDwMaxJobs]; long long ld[kDwMaxJobs]; };
__global__ void dw_reduce_kernel(const float* __restrict__ partial, int splits, int n_jobs, const DwOut o) {
  // one thread = four consecutive columns of one row: 16-byte loads of the (L2-resident) partials, eight splits in flight,
  // every element still summed in split order (bit-identical to the scalar loop)
  const long long total4 = (long long)n_jobs * 16384;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const int job = (int)(i >> 14), rc = (int)(i & 16383) * 4;
    const float4* src = reinterpret_cast<const float4*>(partial + (size_t)job * 65536 + rc);
    const size_t zstride = (size_t)n_jobs * 16384;      // float4 units between splits
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int z = 0;
    for (; z + 8 <= splits; z += 8) {
      float4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = __ldcs(src + (size_t)(z + u) * zstride);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        acc.x += v[u].x;
        acc.y += v[u].y;
        acc.z += v[u].z;
        acc.w += v[u].w;
      }
    }
    for (; z < splits; ++z) {
      const float4 v = __ldcs(src + (size_t)z * zstride);
      acc.x += v.x;
      acc.y += v.y;
      acc.z += v.z;
      acc.w += v.w;
    }
    float* dst = o.ptr[job] + (size_t)(rc >> 8) * o.ld[job] + (rc & 255);      // rows of the rgb-0 / trans-0 gradients are only 8 B aligned
    dst[0] = acc.x;
    dst[1] = acc.y;
    dst[2] = acc.z;
    dst[3] = acc.w;
  }
}

// ------------------------------------------------------------------------------------------ HBM-bound helpers

__device__ __forceinline__ void unpack8(const uint4& q, float f[8]) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    f[2 * e] = __uint_as_float(w[e] << 16);
    f[2 * e + 1] = __uint_as_float(w[e] & 0xffff0000u);
  }
}

// out[m][k] (+ per-block partial) = sum_s thin[s][m] * X[s][k], thin fp32 row-major [S, M<=8], X a tile-image slot.
// thread = (k8 = tid / 8, row group = tid % 8): 16 B image vectors, fp32 accumulate, fixed-order reduction.
template <int M>
__global__ void __launch_bounds__(256) thin_dw_kernel(const float* __restrict__ thin, const uint8_t* __restrict__ images,
                                                      int slot, int n_slots, long long S, long long tiles_per_block,
                                                      float* __restrict__ partial) {
  const long long n_tiles = (S + 127) / 128;
  const long long t0 = blockIdx.x * tiles_per_block, t1 = t0 + tiles_per_block < n_tiles ? t0 + tiles_per_block : n_tiles;
  const int k8 = threadIdx.x >> 3, g = threadIdx.x & 7;
  float acc[M][8];
#pragma unroll
  for (int m = 0; m < M; ++m)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[m][c] = 0.f;
  for (long long t = t0; t < t1; ++t) {
    const uint8_t* img = images + ((size_t)t * n_slots + slot) * kABytes + k8 * 2048;
    for (int i = 0; i < 16; ++i) {
      const int r = g + 8 * i;
      const long long s = t * 128 + r;
      if (s >= S) break;
      float x[8];
      unpack8(*reinterpret_cast<const uint4*>(img + r * 16), x);
#pragma unroll
      for (int m = 0; m < M; ++m) {
        const float w = thin[s * M + m];
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[m][c] = fmaf(w, x[c], acc[m][c]);
      }
    }
  }
#pragma unroll
  for (int m = 0; m < M; ++m)
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float v = acc[m][c];
      v += __shfl_xor_sync(0xffffffffu, v, 1);
      v += __shfl_xor_sync(0xffffffffu, v, 2);
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      if (g == 0) partial[((size_t)blockIdx.x * M + m) * 256 + k8 * 8 + c] = v;
    }
}

// per-ray sums straight from a tile-image slot: out[r][k] = sum over the N samples of ray r of x[s][k].
// One CTA per ray; thread = (k8, row group of 8); rows of one ray are contiguous 16 B vectors inside each tile.
__global__ void __launch_bounds__(256) image_ray_sums_kernel(const uint8_t* __restrict__ images, int slot, int n_slots,
                                                             long long S, int N, float* __restrict__ out) {
  const long long ray = blockIdx.x;
  const int k8 = threadIdx.x >> 3, g = threadIdx.x & 7;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int i = g; i < N; i += 8) {
    const long long s = ray * N + i;
    if (s >= S) break;
    float x[8];
    unpack8(*reinterpret_cast<const uint4*>(images + ((size_t)(s >> 7) * n_slots + slot) * kABytes + k8 * 2048 + (s & 127) * 16), x);
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] += x[c];
  }
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    float v = acc[c];
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    if (g == 0) out[ray * 256 + k8 * 8 + c] = v;
  }
}

// column sums of a thin row-major fp32 matrix [S, C<=8]: partial[block][C]
__global__ void __launch_bounds__(256) thin_colsum_kernel(const float* __restrict__ x, long long S, int C,
                                                          float* __restrict__ partial) {
  __shared__ float sm[8][8];
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < S; s += (long long)gridDim.x * blockDim.x)
    for (int c = 0; c < C; ++c) acc[c] += x[s * C + c];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    float v = acc[c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) sm[w][c] = v;
  }
  __syncthreads();
  if (threadIdx.x < C) {
    float v = 0.f;
    for (int i = 0; i < 8; ++i) v += sm[i][threadIdx.x];
    partial[(size_t)blockIdx.x * C + threadIdx.x] = v;
  }
}

}  // namespace tcb

TP_API int tp_tc_bwd_num_chunks(void) { return tcb::kBwdChunks; }
TP_API int64_t tp_tc_dz_bytes(int64_t S) { return ((S + 127) / 128) * tcb::kDzSlots * (int64_t)tc::kABytes; }
TP_API int tp_tc_dw_splits(int64_t S, int n_jobs) {
  const long long n_tiles = (S + 127) / 128;
  long long splits = tp_num_sms() / (n_jobs < 1 ? 1 : n_jobs);
  if (splits < 1) splits = 1;
  if (splits > n_tiles) splits = n_tiles;
  return (int)splits;
}

TP_API int tp_tc_dw_gemm(const void* a_images, int a_nslots, const void* b_images, int b_nslots, const int32_t* a_slots,
                         const int32_t* b_slots, int n_jobs, int64_t S, float* partial, int64_t partial_floats, void* stream) {
  if (!a_images || !b_images || !partial || !a_slots || !b_slots) return TP_ERR_BAD_ARG;
  if (S < 1 || n_jobs < 1 || n_jobs > tcb::kDwMaxJobs) return TP_ERR_BAD_SHAPE;
  if (((uintptr_t)a_images & 15) || ((uintptr_t)b_images & 15) || ((uintptr_t)partial & 15)) return TP_ERR_ALIGN;
  if (!tp_device_is_sm100()) return TP_ERR_ARCH;
  tcb::DwParams p;
  p.a_images = reinterpret_cast<const uint8_t*>(a_images); p.a_nslots = a_nslots;
  p.b_images = reinterpret_cast<const uint8_t*>(b_images); p.b_nslots = b_nslots;
  for (int j = 0; j < n_jobs; ++j) {
    if (a_slots[j] < 0 || a_slots[j] >= a_nslots || b_slots[j] < 0 || b_slots[j] >= b_nslots) return TP_ERR_BAD_SHAPE;
    p.a_slot[j] = a_slots[j];
    p.b_slot[j] = b_slots[j];
  }
  p.n_jobs = n_jobs; p.splits = tp_tc_dw_splits(S, n_jobs);
  if (partial_floats < (int64_t)p.splits * n_jobs * 65536) return TP_ERR_WORKSPACE;
  p.n_tiles = (S + 127) / 128; p.partial = partial;
  cudaError_t e = cudaFuncSetAttribute(tcb::dw_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)tcb::kDwSmemBytes);
  if (e != cudaSuccess) return (int)e;
  tcb::dw_gemm_kernel<<<p.splits * n_jobs, tcb::kThreads, tcb::kDwSmemBytes, (cudaStream_t)stream>>>(p);
  return tp_launch_status();
}

TP_API int tp_tc_image_ray_sums(const void* images, int slot, int n_slots, int64_t S, int N, float* out, void* stream) {
  if (!images || !out) return TP_ERR_BAD_ARG;
  if (S < 1 || N < 1 || slot < 0 || slot >= n_slots) return TP_ERR_BAD_SHAPE;
  const long long rays = (S + N - 1) / N;
  tcb::image_ray_sums_kernel<<<(unsigned)rays, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint8_t*>(images), slot,
                                                                              n_slots, S, N, out);
  return tp_launch_status();
}

TP_API int tp_thin_colsum(const float* x, int64_t S, int C, float* out, float* workspace, int64_t workspace_floats,
                          void* stream) {
  if (!x || !out || !workspace) return TP_ERR_BAD_ARG;
  if (S < 1 || C < 1 || C > 8) return TP_ERR_BAD_SHAPE;
  int blocks = tp_grid_for(S, 256, 2);
  if (workspace_floats < (int64_t)blocks * C) return TP_ERR_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  tcb::thin_colsum_kernel<<<blocks, 256, 0, st>>>(x, S, C, workspace);
  if (int rc = tp_launch_status()) return rc;
  return tp_reduce_partials(workspace, blocks, C, out, 0, stream);
}

TP_API int tp_tc_thin_dw(const float* thin, int M, const void* images, int slot, int n_slots, int64_t S, float* partial,
                         int64_t partial_floats, int* n_blocks_out, void* stream) {
  if (!thin || !images || !partial) return TP_ERR_BAD_ARG;
  if (S < 1 || slot < 0 || slot >= n_slots || (M != 1 && M != 3 && M != 5)) return TP_ERR_BAD_SHAPE;
  const long long n_tiles = (S + 127) / 128;
  long long blocks = (long long)tp_num_sms() * 4;
  if (blocks > n_tiles) blocks = n_tiles;
  const long long tpb = (n_tiles + blocks - 1) / blocks;
  blocks = (n_tiles + tpb - 1) / tpb;
  if (partial_floats < blocks * M * 256) return TP_ERR_WORKSPACE;
  if (n_blocks_out) *n_blocks_out = (int)blocks;
  const uint8_t* img = reinterpret_cast<const uint8_t*>(images);
  cudaStream_t st = (cudaStream_t)stream;
  if (M == 1) tcb::thin_dw_kernel<1><<<(unsigned)blocks, 256, 0, st>>>(thin, img, slot, n_slots, S, tpb, partial);
  else if (M == 3) tcb::thin_dw_kernel<3><<<(unsigned)blocks, 256, 0, st>>>(thin, img, slot, n_slots, S, tpb, partial);
  else tcb::thin_dw_kernel<5><<<(unsigned)blocks, 256, 0, st>>>(thin, img, slot, n_slots, S, tpb, partial);
  return tp_launch_status();
}

static int fused_grid(long long n_tiles) {
  int grid = tp_num_sms();
  if (n_tiles < grid) grid = (int)n_tiles;
  return grid < 1 ? 1 : grid;
}

TP_API int tp_tc_heads_backward_supported(int64_t S, int64_t per_image) {
  if (S < 1 || per_image < 1) return 0;
  const long long n_tiles = (S + 127) / 128;
  const int grid = fused_grid(n_tiles);
  const long long span = ((n_tiles + grid - 1) / grid) * 128;      // samples of the longest contiguous CTA range
  return (span - 1 + per_image - 1) / per_image + 1 <= tcb::kMaxImagesPerCta ? 1 : 0;
}

TP_API int64_t tp_tc_heads_backward_workspace(int64_t S, int B) {
  const long long n_tiles = (S + 127) / 128;
  const int grid = fused_grid(n_tiles);
  return (int64_t)grid * tcb::kXCols * 256 + (int64_t)grid * 32 + tcb::kXCols * 256 + 8LL * B * 256 +
         (int64_t)tp_tc_dw_splits(S, 6) * 6 * 65536;
}

TP_API int tp_tc_heads_backward(const float* dz_rgb, const float* dz_trans, int64_t S, int N, int64_t per_image, int B,
                                const float* center, const float* ray, const float* depth, int L_view,
                                const void* packed_bwd, const void* saved, void* dz_images, const float* W_r0,
                                int64_t ld_r0, const float* W_t0, int64_t ld_t0, const float* lat_light, int n_light,
                                const float* lat_trans, int n_trans, float* const* grads, float* d_lat_light,
                                float* d_lat_trans, float* workspace, int64_t workspace_floats, void* stream) {
  if (!dz_rgb || !dz_trans || !center || !ray || !depth || !packed_bwd || !saved || !dz_images || !W_r0 || !W_t0 ||
      !lat_light || !lat_trans || !grads || !workspace)
    return TP_ERR_BAD_ARG;
  for (int i = 0; i < 16; ++i)
    if (!grads[i]) return TP_ERR_BAD_ARG;
  if (S < 1 || N < 1 || per_image < 1 || B < 1 || L_view < 0 || L_view > 4 || n_light < 0 || n_light > 64 || n_trans < 0 ||
      n_trans > 64 || (int64_t)B * per_image < S)
    return TP_ERR_BAD_SHAPE;
  const int vc = 3 + 6 * L_view;
  if (ld_r0 < 256 + vc + 3 + n_light || ld_t0 < 256 + n_trans) return TP_ERR_BAD_SHAPE;
  if (!tp_tc_heads_backward_supported(S, per_image)) return TP_ERR_BAD_SHAPE;
  if (((uintptr_t)packed_bwd & 15) || ((uintptr_t)saved & 15) || ((uintptr_t)dz_images & 15) || ((uintptr_t)workspace & 15))
    return TP_ERR_ALIGN;
  if (!tp_device_is_sm100()) return TP_ERR_ARCH;
  if (workspace_floats < tp_tc_heads_backward_workspace(S, B)) return TP_ERR_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const long long n_tiles = (S + 127) / 128;
  const int grid = fused_grid(n_tiles);
  float* extras = workspace;
  float* thin_sums = extras + (size_t)grid * tcb::kXCols * 256;
  float* tot = thin_sums + (size_t)grid * 32;
  float* img = tot + tcb::kXCols * 256;
  float* partial = img + 8 * (size_t)B * 256;

  tcb::FusedParams fp;
  fp.b.dz_rgb = dz_rgb; fp.b.dz_trans = dz_trans; fp.b.S = S;
  fp.b.packed = reinterpret_cast<const uint8_t*>(packed_bwd);
  fp.b.saved = reinterpret_cast<const uint8_t*>(saved);
  fp.b.dz_out = reinterpret_cast<uint8_t*>(dz_images);
  fp.center = center; fp.ray = ray; fp.depth = depth; fp.N = N; fp.per_image = per_image; fp.L_view = L_view;
  fp.extras = extras; fp.thin_sums = thin_sums;
  // debugging aid: a workspace with 2*16*grid extra floats receives the MMA warp's cycle counters in its tail
  const int64_t need = tp_tc_heads_backward_workspace(S, B);
  fp.prof = workspace_floats >= need + 32 * (int64_t)grid ? reinterpret_cast<long long*>(workspace + ((need + 1) & ~(int64_t)1)) : nullptr;
  cudaError_t e = cudaFuncSetAttribute(tcb::backward_chain_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)tcb::kSmemBytesF);
  if (e != cudaSuccess) return (int)e;
  tcb::backward_chain_fused_kernel<<<grid, tcb::kFThreads, tcb::kSmemBytesF, st>>>(fp);
  if (int rc = tp_launch_status()) return rc;

  tcb::FinishParams f;
  f.extras = extras; f.thin_sums = thin_sums; f.grid = grid; f.n_tiles = n_tiles; f.per_image = per_image;
  f.B = B; f.vc = vc; f.n_light = n_light; f.n_trans = n_trans; f.tot = tot; f.img = img;
  f.W_r0 = W_r0; f.ld_r0 = ld_r0; f.W_t0 = W_t0; f.ld_t0 = ld_t0; f.lat_light = lat_light; f.lat_trans = lat_trans;
  for (int i = 0; i < 16; ++i) f.g[i] = grads[i];
  f.d_lat_light = d_lat_light; f.d_lat_trans = d_lat_trans;
  tcb::bwd_finish1_kernel<<<tcb::kXCols, 256, 0, st>>>(f);
  if (int rc = tp_launch_status()) return rc;
  tcb::bwd_finish2_kernel<<<B + 2 * tcb::kFinishParts, 256, 2 * 256 * sizeof(float), st>>>(f);
  if (int rc = tp_launch_status()) return rc;

  // the six 256 x 256 weight gradients: layers 2, 1, 0 of the rgb head, then of the transient head
  tcb::DwParams p;
  p.a_images = reinterpret_cast<const uint8_t*>(dz_images); p.a_nslots = tcb::kDzSlots;
  p.b_images = reinterpret_cast<const uint8_t*>(saved); p.b_nslots = tcb::kFwdSlots;
  const int a_slot[6] = {0, 1, 2, 3, 4, 5}, b_slot[6] = {2, 1, 0, 5, 4, 0};
  for (int j = 0; j < 6; ++j) { p.a_slot[j] = a_slot[j]; p.b_slot[j] = b_slot[j]; }
  p.n_jobs = 6; p.splits = tp_tc_dw_splits(S, 6); p.n_tiles = n_tiles; p.partial = partial;
  e = cudaFuncSetAttribute(tcb::dw_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tcb::kDwSmemBytes);
  if (e != cudaSuccess) return (int)e;
  tcb::dw_gemm_kernel<<<p.splits * 6, tcb::kThreads, tcb::kDwSmemBytes, st>>>(p);
  if (int rc = tp_launch_status()) return rc;
  tcb::DwOut o;
  const int gidx[6] = {4, 2, 0, 12, 10, 8};          // grads[] index of dW2, dW1, dW0 per head
  for (int j = 0; j < 6; ++j) { o.ptr[j] = grads[gidx[j]]; o.ld[j] = 256; }
  o.ld[2] = ld_r0; o.ld[5] = ld_t0;
  for (int j = 6; j < tcb::kDwMaxJobs; ++j) { o.ptr[j] = nullptr; o.ld[j] = 0; }
  tcb::dw_reduce_kernel<<<tp_grid_for(6 * 16384, 256, 4), 256, 0, st>>>(partial, p.splits, 6, o);
  return tp_launch_status();
}
