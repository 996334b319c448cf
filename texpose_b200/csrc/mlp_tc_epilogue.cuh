// Accumulator-drain helpers of the fused forward kernel (mlp_tc.cu):
// TMEM -> registers -> (+bias) ReLU -> bf16 -> SMEM A operand of the next stage, optionally emitting the ReLU bitmask.
#pragma once
#include "mlp_tc_shared.cuh"

namespace tc {

// One 32-column slab of a hidden stage: (+fp32 bias,) ReLU, bf16, store as 4 core-matrix rows of the next A operand.
// kBits (training): also returns the ReLU mask of the 32 columns (bit e = column e is positive) -- one funnel shift per
// element collects the sign bits; the backward reads these 4 KB bitmasks instead of the 64 KB activation tiles.
// kBits also marks the training launch: when `g_dst` is set the same 16-byte groups go straight from the registers to the saved
// tile image in HBM (a warp's store covers 512 contiguous bytes), so the activation save never re-reads the A tile.  The
// stores are streaming (st.global.cs, evict-first): 1.9 GB per C3 step pass through L2 once and must not displace the 2 MB
// weight image every CTA keeps re-reading (measured: 1 130 us with bulk stores -> 1 058 us direct -> 970 us streaming).
template <bool kBias, bool kBits = false>
__device__ __forceinline__ uint32_t hidden_slab(const uint32_t (&v)[32], const float* bias, uint32_t a_dst, uint8_t* g_dst = nullptr) {
  uint32_t signs = 0u;
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    float x[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(v[i + e]);
    if (kBias) {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + i));
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + i + 4));
      x[0] += b0.x; x[1] += b0.y; x[2] += b0.z; x[3] += b0.w;
      x[4] += b1.x; x[5] += b1.y; x[6] += b1.z; x[7] += b1.w;
    }
    if (kBits) {
#pragma unroll
      for (int e = 0; e < 8; ++e) signs = __funnelshift_l(__float_as_uint(x[e]), signs, 1);
    }
    const uint32_t q0 = pack_relu_bf16(x[0], x[1]), q1 = pack_relu_bf16(x[2], x[3]), q2 = pack_relu_bf16(x[4], x[5]),
                   q3 = pack_relu_bf16(x[6], x[7]);
    st_shared_v4(a_dst + (i >> 3) * 2048, q0, q1, q2, q3);
    if (kBits && g_dst) st_global_cs_v4(g_dst + (i >> 3) * 2048, q0, q1, q2, q3);
  }
  return __brev(~signs);      // element 0 was shifted in first: reverse; positive = sign bit clear
}

// Same with the bias row held distributed across the warp (lane l owns columns 4l..4l+3 of the thread's column range, in
// `mine[0]`, and 128+4l.. in `mine[1]` when a thread converts 256 columns): valid when all 32 rows of the warp share one
// bias row (N % 32 == 0).  8 shuffles per 8 columns replace 2 dependent L2 round trips.
template <bool kBits = false>
__device__ __forceinline__ uint32_t hidden_slab_wbias(const uint32_t (&v)[32], const float4 (&mine)[2], int col0, uint32_t a_dst,
                                                      uint8_t* g_dst = nullptr) {
  uint32_t signs = 0u;
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const int c = col0 + i;                       // first column of this group within the thread's range
    const float4 src = mine[(c >> 7) & 1];
    const int l0 = (c & 127) >> 2;
    float x[8];
    x[0] = __uint_as_float(v[i + 0]) + __shfl_sync(0xffffffffu, src.x, l0);
    x[1] = __uint_as_float(v[i + 1]) + __shfl_sync(0xffffffffu, src.y, l0);
    x[2] = __uint_as_float(v[i + 2]) + __shfl_sync(0xffffffffu, src.z, l0);
    x[3] = __uint_as_float(v[i + 3]) + __shfl_sync(0xffffffffu, src.w, l0);
    x[4] = __uint_as_float(v[i + 4]) + __shfl_sync(0xffffffffu, src.x, l0 + 1);
    x[5] = __uint_as_float(v[i + 5]) + __shfl_sync(0xffffffffu, src.y, l0 + 1);
    x[6] = __uint_as_float(v[i + 6]) + __shfl_sync(0xffffffffu, src.z, l0 + 1);
    x[7] = __uint_as_float(v[i + 7]) + __shfl_sync(0xffffffffu, src.w, l0 + 1);
    if (kBits) {
#pragma unroll
      for (int e = 0; e < 8; ++e) signs = __funnelshift_l(__float_as_uint(x[e]), signs, 1);
    }
    const uint32_t q0 = pack_relu_bf16(x[0], x[1]), q1 = pack_relu_bf16(x[2], x[3]), q2 = pack_relu_bf16(x[4], x[5]),
                   q3 = pack_relu_bf16(x[6], x[7]);
    st_shared_v4(a_dst + (i >> 3) * 2048, q0, q1, q2, q3);
    if (kBits && g_dst) st_global_cs_v4(g_dst + (i >> 3) * 2048, q0, q1, q2, q3);
  }
  return __brev(~signs);
}

// Same with the bias row in shared memory (all 128 rows of the tile share it: one ray per tile at N = 128, one image per tile):
// every lane reads the same 16 bytes, i.e. a broadcast ld.shared.v4 -- 2 loads per 8 columns instead of 8 shuffles.  The
// shuffle form costs ~2 000 cycles per table-bias stage (256 warp shuffles per thread against a shuffle unit that serves one
// warp per cycle): 4 % of a super-tile (scripts/fwd_prof.py: the MMA warp waits 2 700 cycles for the stage after each of them).
template <bool kBits = false>
__device__ __forceinline__ uint32_t hidden_slab_sbias(const uint32_t (&v)[32], uint32_t bias_smem, uint32_t a_dst,
                                                      uint8_t* g_dst = nullptr) {
  uint32_t signs = 0u;
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    float4 b0, b1;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b0.x), "=f"(b0.y), "=f"(b0.z), "=f"(b0.w) : "r"(bias_smem + i * 4));
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b1.x), "=f"(b1.y), "=f"(b1.z), "=f"(b1.w) : "r"(bias_smem + i * 4 + 16));
    float x[8];
    x[0] = __uint_as_float(v[i + 0]) + b0.x; x[1] = __uint_as_float(v[i + 1]) + b0.y;
    x[2] = __uint_as_float(v[i + 2]) + b0.z; x[3] = __uint_as_float(v[i + 3]) + b0.w;
    x[4] = __uint_as_float(v[i + 4]) + b1.x; x[5] = __uint_as_float(v[i + 5]) + b1.y;
    x[6] = __uint_as_float(v[i + 6]) + b1.z; x[7] = __uint_as_float(v[i + 7]) + b1.w;
    if (kBits) {
#pragma unroll
      for (int e = 0; e < 8; ++e) signs = __funnelshift_l(__float_as_uint(x[e]), signs, 1);
    }
    const uint32_t q0 = pack_relu_bf16(x[0], x[1]), q1 = pack_relu_bf16(x[2], x[3]), q2 = pack_relu_bf16(x[4], x[5]),
                   q3 = pack_relu_bf16(x[6], x[7]);
    st_shared_v4(a_dst + (i >> 3) * 2048, q0, q1, q2, q3);
    if (kBits && g_dst) st_global_cs_v4(g_dst + (i >> 3) * 2048, q0, q1, q2, q3);
  }
  return __brev(~signs);
}

template <int kSlabs, bool kBits = false>
__device__ __forceinline__ void hidden_epilogue_sbias(uint32_t tmem_d, uint32_t bias_smem, uint32_t a_row,
                                                      uint32_t* words = nullptr, uint8_t* g_row = nullptr) {
  uint32_t va[32], vb[32];
  TP_TMEM_LD32(tmem_d, va);
#pragma unroll
  for (int j = 0; j < kSlabs; j += 2) {
    TP_TMEM_WAIT32(va);
    TP_TMEM_LD32(tmem_d + (j + 1) * 32, vb);
    const uint32_t w0 = hidden_slab_sbias<kBits>(va, bias_smem + j * 128, a_row + j * 4 * 2048, g_row ? g_row + j * 4 * 2048 : nullptr);
    TP_TMEM_WAIT32(vb);
    if (j + 2 < kSlabs) TP_TMEM_LD32(tmem_d + (j + 2) * 32, va);
    const uint32_t w1 = hidden_slab_sbias<kBits>(vb, bias_smem + (j + 1) * 128, a_row + (j + 1) * 4 * 2048,
                                                 g_row ? g_row + (j + 1) * 4 * 2048 : nullptr);
    if (kBits && words) { __stcs(words + j * 128, w0); __stcs(words + (j + 1) * 128, w1); }
  }
}

template <int kSlabs, bool kBits = false>
__device__ __forceinline__ void hidden_epilogue_wbias(uint32_t tmem_d, const float4 (&mine)[2], uint32_t a_row,
                                                      uint32_t* words = nullptr,        // words: plane j at words[j * 128]
                                                      uint8_t* g_row = nullptr) {       // g_row: this row in the saved tile image
  uint32_t va[32], vb[32];
  TP_TMEM_LD32(tmem_d, va);
#pragma unroll
  for (int j = 0; j < kSlabs; j += 2) {
    TP_TMEM_WAIT32(va);
    TP_TMEM_LD32(tmem_d + (j + 1) * 32, vb);
    const uint32_t w0 = hidden_slab_wbias<kBits>(va, mine, j * 32, a_row + j * 4 * 2048, g_row ? g_row + j * 4 * 2048 : nullptr);
    TP_TMEM_WAIT32(vb);
    if (j + 2 < kSlabs) TP_TMEM_LD32(tmem_d + (j + 2) * 32, va);
    const uint32_t w1 = hidden_slab_wbias<kBits>(vb, mine, (j + 1) * 32, a_row + (j + 1) * 4 * 2048,
                                                 g_row ? g_row + (j + 1) * 4 * 2048 : nullptr);
    if (kBits && words) { __stcs(words + j * 128, w0); __stcs(words + (j + 1) * 128, w1); }
  }
}

// Whole 128x256 accumulator row of one thread: TMEM loads are software-pipelined (slab j+1 in flight while slab j is
// converted), ping-ponging two register slabs.
template <bool kBias, int kSlabs, bool kBits = false>
__device__ __forceinline__ void hidden_epilogue(uint32_t tmem_d, const float* bias, uint32_t a_row,
                                                uint32_t* words = nullptr, uint8_t* g_row = nullptr) {
  uint32_t va[32], vb[32];
  TP_TMEM_LD32(tmem_d, va);
#pragma unroll
  for (int j = 0; j < kSlabs; j += 2) {
    TP_TMEM_WAIT32(va);
    TP_TMEM_LD32(tmem_d + (j + 1) * 32, vb);
    const uint32_t w0 = hidden_slab<kBias, kBits>(va, bias + j * 32, a_row + j * 4 * 2048, g_row ? g_row + j * 4 * 2048 : nullptr);
    TP_TMEM_WAIT32(vb);
    if (j + 2 < kSlabs) TP_TMEM_LD32(tmem_d + (j + 2) * 32, va);
    const uint32_t w1 = hidden_slab<kBias, kBits>(vb, bias + (j + 1) * 32, a_row + (j + 1) * 4 * 2048,
                                                  g_row ? g_row + (j + 1) * 4 * 2048 : nullptr);
    if (kBits && words) { __stcs(words + j * 128, w0); __stcs(words + (j + 1) * 128, w1); }
  }
}

}  // namespace tc
