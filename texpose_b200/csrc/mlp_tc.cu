// K2 (bf16 mode): fused per-sample NeRF forward on the 5th-gen tensor cores (tcgen05 + TMEM), sm_100a.
//
// Replaces points_3D -> positional encoding -> 8-layer trunk -> rgb head -> transient head of
// layers/nerf_static_transient_light.py:76-145 (~46 aten kernels and ~30 HBM round trips per chunk in the
// reference) with ONE persistent kernel: activations never leave the SM.
//
// Work decomposition
//   * super-tile = 256 consecutive samples = two M=128 MMA tiles (T0, T1) that march through the 17 GEMM
//     stages in lock-step so every streamed weight chunk is used twice;
//   * per stage and tile:  D[128 x 256 fp32, TMEM] = A[128 x K bf16, SMEM] * W^T[K x 256 bf16, SMEM]
//     issued as tcgen05.mma.cta_group::1.kind::f16 (M=128, N=256 or 16, K=16) by ONE thread;
//   * weights are pre-packed (tp_tc_pack_weights) into the exact SMEM image of each 16 KB K-chunk and
//     streamed through a 4-stage ring with cp.async.bulk (TMA bulk copy) + mbarrier complete_tx;
//   * 8 epilogue warps (one TMEM lane quarter each, 4 per tile): tcgen05.ld -> +bias -> ReLU -> bf16 ->
//     st.shared straight into the K-major core-matrix layout the next stage's A descriptor reads;
//   * per-ray constants (view-direction encoding, light latent) and per-image constants (transient latent)
//     are folded into fp32 biases, so they cost no MMA work per sample: per-image rows by a tiny pre-kernel, the per-ray
//     row by a pre-kernel table (per-sample launches) or by the tile's own warps (render launch);
//   * render launch (tp_render_fused_forward, Graph.render model/nerf_adapt_st_gan.py:565-631 as ONE kernel): the tile's
//     rows generate their ray from the pixel index, their sample depth from the ray's bounds (midpoint / injected rand /
//     Philox), and the last stage's epilogue composites the tile's rays (row = sample: warp scan + cross-warp carry) --
//     no depth, bias-table, rgb or uncertainty tensor ever exists in HBM; per ray 8 B in, 56 B out (+ 16 B per sample for
//     the API's alpha / density tensors);
//   * the trunk feature (needed by both heads) is parked in an L2-resident scratch with a bulk store after
//     the last trunk layer and bulk-loaded back before the transient head.
//
// SMEM (bytes): A0 64K | A1 64K | E0 16K | E1 16K | ring 4x16K | barriers 128 | compositing scratch 544 | bias rows 2 x 1K = 232 096 (<= 227 KB).
// TMEM: 512 columns = two 128x256 fp32 accumulators.
//
// Operand layout (no swizzle, K-major "interleave" canonical layout): element (row r, col k) of a tile with
// `rows` rows lives at  (k/8)*rows*16 + r*16 + (k%8)*2  bytes -> 8x8 core matrices of 128 contiguous bytes,
// LBO (K-direction core-matrix stride) = rows*16, SBO (8-row-group stride) = 128.
#include "mlp_tc_shared.cuh"
#include "mlp_tc_epilogue.cuh"
#include "../../include/texpose_b200.h"

namespace tc {

// 8 epilogue warps (one per tile and TMEM lane quarter: 256 accumulator columns per thread), then one TMA producer warp and one
// MMA issuer warp
constexpr int kEpiWarps = 8, kProducerWarp = kEpiWarps, kMmaWarp = kEpiWarps + 1, kThreads = (kEpiWarps + 2) * 32;
constexpr int kStages = 4;
constexpr uint32_t kOffA = 0, kOffE = 2 * kABytes, kOffRing = kOffE + 2 * kEBytes;
constexpr uint32_t kOffBar = kOffRing + kStages * kChunkBytes;
// compositing scratch of the render launch: [tile 2][ warp totals 4 x 3 | warp partial sums 4 x 14 ] floats, then one 1 KB
// fp32 bias row per tile (the per-ray / per-image row of the two table-bias stages when all 128 rows of the tile share it)
constexpr int kCompFloats = 4 * 3 + 4 * 14;
constexpr uint32_t kOffComp = kOffBar + 128;
constexpr uint32_t kOffBias = kOffComp + 2 * kCompFloats * 4;
constexpr uint32_t kSmemBytes = kOffBias + 2 * 1024;
static_assert(kOffBias % 16 == 0, "bias rows are read with ld.shared.v4");
static_assert(kSmemBytes <= 232448, "227 KB of shared memory per CTA");
constexpr unsigned kFullMask = 0xffffffffu;
constexpr int kViewBiasLayer = 6;      // render launch: the view-direction bias rows are computed while this stage's MMAs run

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
  return v;
}
__device__ __forceinline__ float warp_scan(float v, int lane) {      // inclusive
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float n = __shfl_up_sync(kFullMask, v, o);
    if (lane >= o) v += n;
  }
  return v;
}

// ------------------------------------------------------------------------------------------ fused render pieces (mode 3)
// One sample of the render launch: its ray is generated from the pixel index (camera.py:292-314, same arithmetic as
// tp_raygen), its depth from the ray's bounds (model/nerf_adapt_st_gan.py:682-700, same arithmetic and Philox stream as
// tp_sample_depth), the interval to the next sample of the ray for the compositing, and its encoding goes into the E tile.
struct RenderSample {
  long long ray;      // ray index within the launch (clamped to the last ray for dead rows)
  int k;              // sample index within the ray
  int img;            // view
  float d, dist;      // depth, (d_{k+1} - d_k) * |ray|  (1e10 * |ray| for the last sample: layers/..light.py:169-175)
  float dir[3];       // ray direction (unnormalised, camera-z = 1)
  float xyz[3];       // the sample point c + ray * d
  bool live;
};

// Stratified jitter of this lane's sample and of the NEXT sample of its ray (for the interval).  A warp holds 32 consecutive
// samples = 8 Philox quads (tp_sample_depth's stream: one Philox4x32-10 block per 4 consecutive samples, counter = sample / 4):
// lanes 0..8 evaluate quads 0..8 of the warp ONCE (quad 8 = the first sample of the next warp, lane 31's neighbour) and four
// shuffles hand every lane its component -- one Philox evaluation per warp instead of two.
__device__ __forceinline__ void render_jitter_pair(const Params& p, long long s, int lane, bool has_next, float& u0, float& u1) {
  if (p.depth_mode == 1) {
    u0 = u1 = 0.5f;
    return;
  }
  if (p.depth_mode == 0) {
    u0 = p.rand[s];
    u1 = __shfl_down_sync(kFullMask, u0, 1);
    if (lane == 31 && has_next) u1 = p.rand[s + 1];
    return;
  }
  const long long qd = ((s - lane) >> 2) + lane;      // (s - lane) is the warp's first sample: a multiple of 32
  const uint4 x = tp_philox((uint32_t)qd, (uint32_t)(qd >> 32), (uint32_t)p.seed, (uint32_t)(p.seed >> 32));
  const int src = lane >> 2, e = lane & 3;
  const float c0 = __shfl_sync(kFullMask, tp_u01(x.x), src), c1 = __shfl_sync(kFullMask, tp_u01(x.y), src),
              c2 = __shfl_sync(kFullMask, tp_u01(x.z), src), c3 = __shfl_sync(kFullMask, tp_u01(x.w), src);
  u0 = e == 0 ? c0 : e == 1 ? c1 : e == 2 ? c2 : c3;
  const float nq = __shfl_sync(kFullMask, tp_u01(x.x), 8);      // first component of the next warp's first quad
  u1 = __shfl_down_sync(kFullMask, u0, 1);
  if (lane == 31) u1 = nq;
}

// stratified_depth for N = 2^m: (u + k) / N is an exact scaling, so the multiplication gives the division's bits
__device__ __forceinline__ float stratified_depth_pow2(float u, int k, float inv_n, float lo, float hi) {
  return __fadd_rn(__fmul_rn(__fmul_rn(__fadd_rn(u, (float)k), inv_n), __fsub_rn(hi, lo)), lo);
}

// pixel b, pix -> ray, bounds, jitter (key s), depth, interval, point of a sample whose k, ray, live and img are set
__device__ __forceinline__ void render_fetch_at(const Params& p, long long b, long long pix, long long s, int lane, RenderSample& o) {
  const int N = p.N;
  float c[3];
  unproject(p.kinv + b * 9, p.pinv + b * 12, __fadd_rn((float)(pix % p.W), p.pix_offset),
            __fadd_rn((float)(pix / p.W), p.pix_offset), c, o.dir);
  const long long zi = b * (long long)p.H * p.W + pix;
  const float lo = p.z_near[zi], hi = p.z_far[zi];
  float u0, u1;
  render_jitter_pair(p, s, lane, o.k + 1 < N, u0, u1);
  const float inv_n = 1.f / (float)N;                      // N in {32, 64, 128}: exact
  o.d = stratified_depth_pow2(u0, o.k, inv_n, lo, hi);
  const float dn = stratified_depth_pow2(u1, o.k + 1, inv_n, lo, hi);
  const float len = sqrtf(o.dir[0] * o.dir[0] + o.dir[1] * o.dir[1] + o.dir[2] * o.dir[2]);
  o.dist = __fmul_rn(o.k + 1 < N ? __fsub_rn(dn, o.d) : 1e10f, len);
#pragma unroll
  for (int j = 0; j < 3; ++j) o.xyz[j] = __fadd_rn(c[j], __fmul_rn(o.dir[j], o.d));      // camera.py:317-322
}
// Everything of a sample but its encoding: pixel -> ray, bounds, jitter, depth, interval, point.  A call, like the other render
// pieces: the stage loop of the epilogue warps must stay small and spill-free -- local-memory traffic and instruction fetch share
// the SM's data paths with the MMAs' operand reads, and every build that carried this code inside the loop was slower
// (scripts/fwd_prof.py).  It runs where both tiles and the tensor pipe wait anyway (below); the encoding follows from `xyz`.
__device__ __noinline__ RenderSample render_fetch(const Params& p, long long tile, int row, int lane) {
  RenderSample o;
  const int N = p.N;                                      // divides 128: a tile holds 128 / N whole rays
  o.k = row % N;
  const long long n_rays = p.S / N, ray_raw = tile * (128 / N) + row / N;
  o.live = ray_raw < n_rays;
  o.ray = o.live ? ray_raw : n_rays - 1;
  const long long s = o.ray * N + o.k;
  const long long b = o.ray / p.R;
  o.img = (int)b;
  const long long pix = p.ray_idx ? p.ray_idx[o.ray] : p.ray0 + (o.ray - b * p.R);
  render_fetch_at(p, b, pix, s, lane, o);
  return o;
}
// List mode (kMode 4): ray j of the launch is slot j of the object-pixel list, entry q = view * HW + pixel; a pad entry ~(view * HW)
// is rendered as pixel 0 of its view and stores nothing.  The sample's key -- its jitter and its output address -- is q * N + k: the
// key a full-frame launch (ray_idx NULL, ray0 = 0, R = HW) gives the same pixel's sample, so the two render it bit for bit alike.
__device__ __noinline__ RenderSample render_fetch_list(const Params& p, long long tile, int row, int lane) {
  RenderSample o;
  const int N = p.N;
  o.k = row % N;
  const long long q = p.list[tile * (128 / N) + row / N], HW = (long long)p.H * p.W;
  o.live = q >= 0;
  o.ray = o.live ? q : ~q;      // the frame position the outputs are stored at
  const long long b = o.ray / HW;
  o.img = (int)b;
  render_fetch_at(p, b, o.ray - b * HW, o.ray * N + o.k, lane, o);
  return o;
}
// first (end = 0) / one past the last (end = 1) super-tile of this rank's share of the list: rank r of w takes
// [floor(r T / w), floor((r + 1) T / w)), T = n_slots / (256 / N)
__device__ __forceinline__ long long list_shard(const Params& p, int end) {
  return *p.n_slots / (256 / p.N) * (p.shard_rank + end) / p.shard_world;
}
__device__ __noinline__ void render_encode(const float x, const float y, const float z, uint32_t e_smem, int row) {
  const float xyz[3] = {x, y, z};
  uint32_t e[32];
  encode_xyz_regs(xyz, e);
  store_encoding(e, e_smem, row);
}

// rgb-0 bias row of a ray: imgbias_rgb[view] + W_view [u, enc(u)], u = ray / |ray| (layers/..light.py:104-117,155-157).  Same
// operation order as tp_tc_ray_bias, whose 315 MB table this replaces (one fma chain per column, inputs in ascending order), so
// the row has the table's bits.  The ray's N / 32 warps share the row: warp w computes columns [w, w+1) * 256 / wpr, every lane
// kC = 8 / wpr consecutive ones; lane j holds element j of the 3+6L encoding and shuffles broadcast it.  The 27 inputs are taken
// nine at a time in the shadow of three consecutive trunk stages (the nine weight loads of a batch are independent: one L2
// round trip per stage, 18-36 registers), the partial sums wait in registers, and the slices meet in a 1 KB slot of the CTA's
// L2-resident scratch; at the rgb-0 stage the ray's warps read the row back exactly as the per-sample launches read the table.
__device__ __noinline__ float render_view_element(const Params& p, const RenderSample& rs, int lane) {
  const float len = unit_length(rs.dir[0], rs.dir[1], rs.dir[2]);
  const int L = p.L_view, vc = 3 + 6 * L;
  float e = 0.f;
  if (lane < vc) {
    const int jj = lane - 3, cc = lane < 3 ? lane : jj / (2 * L);
    const float uc = __fdiv_rn(cc == 0 ? rs.dir[0] : cc == 1 ? rs.dir[1] : rs.dir[2], len);
    e = uc;
    if (lane >= 3) {
      const int rem = jj - cc * 2 * L, k = rem < L ? rem : rem - L;
      const float arg = __fmul_rn(uc, ldexpf(3.14159265358979323846f, k));
      e = rem < L ? sinf(arg) : cosf(arg);
    }
  }
  return e;
}
// inputs j0 .. j0+8 of columns col .. col+kC-1 (kC = 2 or 4): acc[c] = fma(W[j][col+c], e_j, acc[c]) in ascending j.  A call,
// not inlined (the stage loop of the epilogue warps stays small; arguments and result travel in registers).
template <int kC>
__device__ __noinline__ float4 render_view_batch(const Params& p, float e, int col, int j0, float4 acc4) {
  const int vc = 3 + 6 * p.L_view;
  float acc[4] = {acc4.x, acc4.y, acc4.z, acc4.w};
  float w[9][kC];
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    if (j0 + i < vc) {
      const float* wr = p.wview + (j0 + i) * 256 + col;
      if (kC == 2) {
        const float2 t2 = __ldg(reinterpret_cast<const float2*>(wr));
        w[i][0] = t2.x; w[i][1] = t2.y;
      } else {
        const float4 t4 = __ldg(reinterpret_cast<const float4*>(wr));
        w[i][0] = t4.x; w[i][1] = t4.y; w[i][kC - 2] = t4.z; w[i][kC - 1] = t4.w;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    const float ej = __shfl_sync(kFullMask, e, (j0 + i) & 31);
    if (j0 + i < vc) {
#pragma unroll
      for (int c = 0; c < kC; ++c) acc[c] = fmaf(w[i][c], ej, acc[c]);
    }
  }
  return make_float4(acc[0], acc[1], acc[2], acc[3]);
}

// Compositing of the tile's rays as the epilogue of the last stage (layers/nerf_static_transient_light.py:168-212, SURVEY
// appendix C; arithmetic of csrc/composite.cu): row = sample, so the three exclusive cumulative sums are a warp scan plus the
// totals of the ray's earlier warps (N / 32 warps per ray, exchanged through `sc`), and the 14 per-ray sums a warp reduction
// plus the same exchange.  Per sample it writes alpha_static, alpha_transient and density (16 B), per ray 14 floats.
__device__ __noinline__ void render_composite(const Params& p, float* sc, int t, int q, int lane, long long ray, int k, float d_k,
                                              float dist, bool live, float sig_s, float sig_t, float cs0, float cs1, float cs2,
                                              float ct0, float ct1, float ct2, float u) {
  struct { long long ray; int k; float d, dist; bool live; } rs = {ray, k, d_k, dist, live};
  const float cs[3] = {cs0, cs1, cs2}, ct[3] = {ct0, ct1, ct2};
  float* tot = sc;             // [4 warps][3]
  float* red = sc + 12;        // [4 warps][14]
  const float sd_s = __fmul_rn(sig_s, rs.dist), sd_t = __fmul_rn(sig_t, rs.dist), sd = __fadd_rn(sd_s, sd_t);
  const float in_j = warp_scan(sd, lane), in_s = warp_scan(sd_s, lane), in_t = warp_scan(sd_t, lane);
  if (lane == 31) {
    tot[q * 3] = in_j;
    tot[q * 3 + 1] = in_s;
    tot[q * 3 + 2] = in_t;
  }
  const float pj = __shfl_up_sync(kFullMask, in_j, 1), ps_ = __shfl_up_sync(kFullMask, in_s, 1), pt_ = __shfl_up_sync(kFullMask, in_t, 1);
  named_bar_sync(1 + t, 128);
  const int wpr = p.N >> 5, q0 = q & ~(wpr - 1);      // warps per ray (1, 2, 4), first warp of this ray
  float ex_j = lane ? pj : 0.f, ex_s = lane ? ps_ : 0.f, ex_t = lane ? pt_ : 0.f;
  {
    float cj = 0.f, c_s = 0.f, c_t = 0.f;
    for (int w = q0; w < q; ++w) {
      cj += tot[w * 3];
      c_s += tot[w * 3 + 1];
      c_t += tot[w * 3 + 2];
    }
    ex_j += cj;
    ex_s += c_s;
    ex_t += c_t;
  }
  const float Es = expf(-sd_s), Et = expf(-sd_t), E = expf(-sd);
  const float T = expf(-ex_j), Ts = expf(-ex_s), Tt = expf(-ex_t);
  const float as = 1.f - Es, at = 1.f - Et, a = 1.f - E;
  const float w_ps = T * as, w_pt = T * at, w_p = T * a, w_qs = Ts * as, w_qt = Tt * at;
  float acc[14];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    acc[c] = cs[c] * w_ps + ct[c] * w_pt;
    acc[3 + c] = w_qs * cs[c];
    acc[6 + c] = w_qt * ct[c];
  }
  acc[9] = rs.d * w_qs;
  acc[10] = w_p;
  acc[11] = w_qs;
  acc[12] = w_qt;
  acc[13] = u * w_pt;
  // warp totals of the 14 (padded to 16) sums by recursive halving: at every step a lane keeps one half of its values and adds
  // the partner's -- 8 + 4 + 2 + 1 + 1 = 16 shuffles instead of 14 x 5; lane l ends up with the total of value (l >> 1) & 15... see idx
  float v16[16];
#pragma unroll
  for (int i = 0; i < 14; ++i) v16[i] = acc[i];
  v16[14] = v16[15] = 0.f;
  float v8[8], v4[4], v2[2];
  {
    const bool up = (lane & 16) != 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float send = up ? v16[i] : v16[i + 8];
      const float recv = __shfl_xor_sync(kFullMask, send, 16);
      v8[i] = (up ? v16[i + 8] : v16[i]) + recv;
    }
  }
  {
    const bool up = (lane & 8) != 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float send = up ? v8[i] : v8[i + 4];
      const float recv = __shfl_xor_sync(kFullMask, send, 8);
      v4[i] = (up ? v8[i + 4] : v8[i]) + recv;
    }
  }
  {
    const bool up = (lane & 4) != 0;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const float send = up ? v4[i] : v4[i + 2];
      const float recv = __shfl_xor_sync(kFullMask, send, 4);
      v2[i] = (up ? v4[i + 2] : v4[i]) + recv;
    }
  }
  float v1;
  {
    const bool up = (lane & 2) != 0;
    const float send = up ? v2[0] : v2[1];
    const float recv = __shfl_xor_sync(kFullMask, send, 2);
    v1 = (up ? v2[1] : v2[0]) + recv;
  }
  v1 += __shfl_xor_sync(kFullMask, v1, 1);
  // value index held by this lane: bit 4 of the lane chose +8, bit 3 +4, bit 2 +2, bit 1 +1
  const int vidx = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
  if ((lane & 1) == 0 && vidx < 14) red[q * 14 + vidx] = v1;
  if (rs.live) {
    const long long s = rs.ray * p.N + rs.k;
    if (p.o_as) __stcs(p.o_as + s, as);
    if (p.o_at) __stcs(p.o_at + s, at);
    if (p.density) __stcs(reinterpret_cast<float2*>(p.density) + s, make_float2(sig_s, sig_t));
  }
  named_bar_sync(1 + t, 128);
  if (q == q0 && lane < 14 && rs.live) {
    float v = 0.f;
    for (int w = q0; w < q0 + wpr; ++w) v += red[w * 14 + lane];
    const long long r = rs.ray;
    float* dst = lane < 3 ? (p.o_rgb ? p.o_rgb + r * 3 + lane : nullptr)
               : lane < 6 ? (p.o_rgb_s ? p.o_rgb_s + r * 3 + lane - 3 : nullptr)
               : lane < 9 ? (p.o_rgb_t ? p.o_rgb_t + r * 3 + lane - 6 : nullptr)
               : lane == 9 ? (p.o_depth ? p.o_depth + r : nullptr)
               : lane == 10 ? (p.o_op ? p.o_op + r : nullptr)
               : lane == 11 ? (p.o_op_s ? p.o_op_s + r : nullptr)
               : lane == 12 ? (p.o_op_t ? p.o_op_t + r : nullptr)
                            : (p.o_unc ? p.o_unc + r : nullptr);
    if (lane == 13) v += p.min_uncert;
    if (dst) *dst = v;
  }
}

// kNL: number of stages run (kNumLayers = all; kStaticLayers = static-only rendering).  A template parameter, not a field of
// Params: a run-time stage count costs 0.3 ms per C2 frame (same-box A/B).
// kMode: 0 = general (any N: the per-sample launches, with or without the activation save, whose N is not a multiple of 32);
// 1 = the plain inference launch (per-sample outputs, no activation save); 2 = the plain training launch (activation save + ReLU
// bitmasks); 3 = the fused render launch (rays, depths, view bias and compositing in-kernel; per-ray outputs); 4 = the render launch
// over an object-pixel list, sharded over the ranks of a frame (render_fetch_list, list_shard).  Modes 1-4 are launched only when
// N % 32 == 0 and compile the branches of the other launch kinds out.
// kSmemBias: the launch has one ray per tile (N = 128, hence also one image per tile): the per-ray / per-image bias row of the
// two table-bias stages sits in shared memory and the drain reads it with broadcast loads instead of warp shuffles.
template <int kNL = kNumLayers, int kMode = 0, bool kSmemBias = false>
// (320 threads allocate registers as 12 warps -- warps are allocated in fours -- so the cap is 168 registers per thread; the render
// launch keeps its look-ahead state (next sample's encoding, finished sample) partly in local memory: a few dozen L1-resident
// STL / LDL per super-tile, cheaper than recomputing it on the critical path)
__global__ void __launch_bounds__(kThreads, 1) nerf_stl_forward_kernel(const Params p) {
  constexpr bool kRender = kMode >= 3, kList = kMode == 4;
  static_assert(!kSmemBias || kMode != 0, "shared-memory bias rows: launches with N % 32 == 0 only");
  uint8_t* const p_save = (kMode == 1 || kRender) ? nullptr : p.save;
  constexpr int kTileThreads = 128;     // epilogue threads working on one tile
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // provably warp-uniform role index
  const int lane = threadIdx.x & 31;
  // barriers
  const uint32_t bar0 = sbase + kOffBar;
  auto bar_full = [&](int s) { return bar0 + 8 * s; };
  auto bar_empty = [&](int s) { return bar0 + 8 * (kStages + s); };
  auto bar_acc = [&](int t) { return bar0 + 8 * (2 * kStages + t); };
  auto bar_ready = [&](int t) { return bar0 + 8 * (2 * kStages + 2 + t); };
  auto bar_reload = [&](int t) { return bar0 + 8 * (2 * kStages + 4 + t); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffBar + 8 * (2 * kStages + 6));

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_empty(s), 1);
    }
    for (int t = 0; t < 2; ++t) {
      mbar_init(bar_acc(t), 1);
      mbar_init(bar_ready(t), kTileThreads / 32);     // one arrive per epilogue warp of the tile
      mbar_init(bar_reload(t), 1);
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {   // TMEM: all 512 columns (one CTA per SM)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // super-tiles of the launch; list mode: of this rank's share, whose first one is super-tile st0 of the list
  const long long n_super = kList ? list_shard(p, 1) - list_shard(p, 0) : (p.S + 255) / 256;

  if (warp == kProducerWarp) {
    // ================================================================ weight producer (converged warp, one lane issues)
    {
      uint32_t stage = 0, phase = 0;
      for (long long st = blockIdx.x; st < n_super; st += gridDim.x) {
        int c = 0;
        for (int L = 0; L < kNL; ++L) {
          const Layer ly = kLayers[L];
          const int nch = ly.small ? 1 : ly.a_chunks + ly.e_chunks + ly.bias_chunk;
          for (int j = 0; j < nch; ++j, ++c) {
            // full 16 KB K=32 chunks; the N=16 chunk and the bias chunk only carry 8 KB
            const uint32_t bytes = (ly.small || j >= ly.a_chunks + ly.e_chunks) ? kChunkBytes / 2 : kChunkBytes;
            mbar_wait(bar_empty(stage), phase ^ 1);
            if (elect_one_sync()) {
              mbar_expect_tx(bar_full(stage), bytes);
              bulk_g2s(sbase + kOffRing + stage * kChunkBytes, p.packed + (size_t)c * kChunkBytes, bytes, bar_full(stage));
            }
            __syncwarp();
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ================================================================ MMA issuer (converged warp, one lane issues)
    // Inside a stage tile 0 runs one weight chunk ahead of tile 1 (both still consume every chunk from the same ring slot):
    // T0's accumulator completes 512 cycles before T1's, so T0's epilogue -- and T0's first MMAs of the next stage -- overlap
    // T1's MMAs / epilogue instead of leaving the tensor pipe idle.
    {
      uint32_t chunk_base = 0, ready_ph = 0, reload_ph = 0;   // per-tile phase bits (bit t)
#ifdef TP_FWD_PROF
      long long pf_ready[2][kNumLayers] = {}, pf_full[kNumLayers] = {}, pf_total = 0;
      const long long pf_t0 = clock64();
#endif
      const uint32_t idesc256 = umma_idesc(128, 256), idesc16 = umma_idesc(128, 16);
      constexpr uint32_t kHi = (128u >> 4) | (1u << 14);   // SBO = 128 B, descriptor version 1
      for (long long st = blockIdx.x; st < n_super; st += gridDim.x) {
        for (int L = 0; L < kNL; ++L) {
          const Layer ly = kLayers[L];
          const int nch = ly.small ? 1 : ly.a_chunks + ly.e_chunks + ly.bias_chunk;
          for (int step = 0; step <= nch; ++step) {
#pragma unroll
            for (int t = 0; t < 2; ++t) {
              const int c = step - t;
              if (c < 0 || c >= nch) continue;
              const uint32_t abs_chunk = chunk_base + c;
              const uint32_t stage = abs_chunk % kStages, phase = (abs_chunk / kStages) & 1u;
#ifdef TP_FWD_PROF
              const long long pf_a = clock64();
#endif
              if (t == 0) mbar_wait(bar_full(stage), phase);          // first touch of this ring slot
#ifdef TP_FWD_PROF
              const long long pf_b = clock64();
              pf_full[L] += pf_b - pf_a;
#endif
              if (c == 0) {
                mbar_wait(bar_ready(t), (ready_ph >> t) & 1u);
#ifdef TP_FWD_PROF
                pf_ready[t][L] += clock64() - pf_b;
#endif
                ready_ph ^= 1u << t;
                if (ly.reload) {
                  mbar_wait(bar_reload(t), (reload_ph >> t) & 1u);
                  reload_ph ^= 1u << t;
                }
              }
              tc_fence_after();
              const uint32_t wsm = sbase + kOffRing + stage * kChunkBytes;
              const uint32_t d_tmem = tmem_base + t * 256;
              if (elect_one_sync()) {
                // descriptor words: lo = start>>4 | (LBO>>4)<<16, hi = SBO>>4 | version(1)<<14
                if (ly.small) {
                  // one chunk = [32 k8][16 rows][8]: 16 K-steps over the full K=256 of A_t
                  uint32_t a_lo = ((sbase + kOffA + t * kABytes) >> 4) | ((2048u >> 4) << 16);
                  uint32_t b_lo = (wsm >> 4) | ((256u >> 4) << 16);
#pragma unroll
                  for (int ks = 0; ks < 16; ++ks) {
                    umma_bf16_lohi(d_tmem, a_lo, kHi, b_lo, kHi, idesc16, ks > 0 ? 1u : 0u);
                    a_lo += 4096u >> 4;
                    b_lo += 512u >> 4;
                  }
                } else if (c >= ly.a_chunks + ly.e_chunks) {
                  // bias step: A = E columns 48..63 (column 63 == 1), B = [2 k8][256 rows][8], zero except the bias column
                  const uint32_t a_lo = ((sbase + kOffE + t * kEBytes + 6 * 2048) >> 4) | ((2048u >> 4) << 16);
                  const uint32_t b_lo = (wsm >> 4) | ((4096u >> 4) << 16);
                  umma_bf16_lohi(d_tmem, a_lo, kHi, b_lo, kHi, idesc256, 1u);
                } else {
                  const bool from_e = c >= ly.a_chunks;
                  const uint32_t a0 = from_e ? sbase + kOffE + t * kEBytes + (c - ly.a_chunks) * 4 * 2048
                                             : sbase + kOffA + t * kABytes + c * 4 * 2048;
                  const uint32_t a_lo = (a0 >> 4) | ((2048u >> 4) << 16);
                  const uint32_t b_lo = (wsm >> 4) | ((4096u >> 4) << 16);
                  umma_bf16_lohi(d_tmem, a_lo, kHi, b_lo, kHi, idesc256, c > 0 ? 1u : 0u);
                  umma_bf16_lohi(d_tmem, a_lo + (4096u >> 4), kHi, b_lo + (8192u >> 4), kHi, idesc256, 1u);
                }
                if (c == nch - 1) umma_commit(bar_acc(t));       // accumulator of tile t complete
                if (t == 1) umma_commit(bar_empty(stage));       // ring slot reusable once both tiles' MMAs retire
              }
              __syncwarp();
            }
          }
          chunk_base += nch;
        }
      }
#ifdef TP_FWD_PROF
      if (lane == 0) {      // [CTA][tile][stage][4]: cycles waiting for the tile's epilogue, for a weight chunk (tile 0), total, super-tiles
        long long* o = reinterpret_cast<long long*>(p.scratch + (size_t)p.prof_offset) + (size_t)blockIdx.x * 2 * kNumLayers * 4;
        long long n_st = 0;
        for (long long st = blockIdx.x; st < n_super; st += gridDim.x) ++n_st;
        pf_total = clock64() - pf_t0;
        for (int t = 0; t < 2; ++t)
          for (int L = 0; L < kNumLayers; ++L) {
            long long* r = o + (t * kNumLayers + L) * 4;
            r[0] = pf_ready[t][L]; r[1] = t == 0 ? pf_full[L] : 0; r[2] = pf_total; r[3] = n_st;
          }
      }
#endif
    }
  } else {
    // ================================================================ encode + epilogue warps
    // warp -> (TMEM lane quarter q = warp % 4, tile t): a thread owns one row of its tile, all 256 accumulator columns
    const int q = warp & 3, t = (warp >> 2) & 1, row = q * 32 + lane;
    const uint32_t a_smem = sbase + kOffA + t * kABytes, e_smem = sbase + kOffE + t * kEBytes;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16) + t * 256;
    uint8_t* my_scratch = p.scratch + ((size_t)blockIdx.x * 2 + t) * kABytes;
    // render launch: view-bias rows of this tile's rays (<= 4 rays x 1 KB), behind the parked features of all CTAs
    float* vb_slot = reinterpret_cast<float*>(p.scratch + (size_t)gridDim.x * 2 * kABytes) + ((size_t)blockIdx.x * 2 + t) * 4 * 256;
    uint32_t acc_ph = 0;
    // all 32 rows of a warp share the ray (and image) when N is a multiple of 32; tail rows are clamped to the last
    // sample, which then belongs to the same ray as the warp's live rows
    const bool warp_bias = kMode ? true : (p.N % 32 == 0);      // modes 1-3 are launched only when N % 32 == 0
    bool store_pending = false;      // a bulk store of A_t (feature park / activation save) may still be reading it
    RenderSample rs = {}, nxt = {};          // render launch: the sample this row holds / will hold in the next super-tile
    // ... and the finished sample of the previous super-tile: composited where both tiles and the tensor pipe wait anyway
    long long done_ray = 0;
    int done_k = 0;
    float done_d = 0.f, done_dist = 0.f, done_v[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    bool done_live = false, have_done = false;
    uint32_t enc_next[32];                   // per-sample launches: the next sample's encoding, computed a stage early (below)
    float4 vb_acc = make_float4(0.f, 0.f, 0.f, 0.f);         // view-direction bias of the tile's ray(s): partial sums across three stages
    float vb_e = 0.f;
    int iter = 0;
    for (long long st = blockIdx.x; st < n_super; st += gridDim.x, ++iter) {
      const long long s_raw = (st * 2 + t) * 128 + row;
      const bool live = s_raw < p.S;
      const long long s = live ? s_raw : p.S - 1;
      if (!kRender || iter == 0) {     // (the render launch encodes the next super-tile at the end of the last stage, below)
        if (kRender) {
          if constexpr (kList) rs = render_fetch_list(p, (list_shard(p, 0) + st) * 2 + t, row, lane);
          else rs = render_fetch(p, st * 2 + t, row, lane);
          render_encode(rs.xyz[0], rs.xyz[1], rs.xyz[2], e_smem, row);
        } else if (kMode == 0 || iter == 0) {
          encode_sample(p, s, e_smem, row);
        } else {
          store_encoding(enc_next, e_smem, row);      // worked out during the previous super-tile (below)
        }
        fence_proxy_async_smem();
        tc_fence_before();
        __syncwarp();                    // every lane's st.shared + proxy fence precede the warp's single arrive
        if (lane == 0) mbar_arrive(bar_ready(t));
      }

      float sigma_s = 0.f, rgb_s[3] = {0.f, 0.f, 0.f};
      for (int L = 0; L < kNL; ++L) {
        const Layer ly = kLayers[L];
        // table biases (per ray / per image): when every row of this warp shares the bias row, each lane fetches its
        // float4 slice(s) now -- the L2 latency hides behind the MMAs of this stage.  The render launch computes the per-ray
        // row here instead of reading a table.
        float4 wb[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
        const bool table_bias = ly.epi == EPI_HIDDEN && ly.bias_kind != BIAS_MMA;
        const uint32_t bias_sm = sbase + kOffBias + t * 1024;
        // the render launch has produced its per-ray row in place (below); every other table row is copied in here
        const bool copy_row = kSmemBias && table_bias && !(kRender && ly.bias_kind == BIAS_RAY);
        if (copy_row) {
          // 128 threads x 8 bytes: the tile's bias row -> shared memory (the loads fly during the stage's MMAs)
          const long long img = kRender ? (long long)rs.img : s / p.per_image;
          const float* brow = ly.bias_kind == BIAS_RAY ? p.raybias + (s / p.N) * 256 : p.imgbias + img * 256;
          const float2 b2 = __ldg(reinterpret_cast<const float2*>(brow) + row);
          asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(bias_sm + row * 8), "f"(b2.x), "f"(b2.y) : "memory");
        } else if (table_bias && warp_bias && !kSmemBias) {
          if (kRender && ly.bias_kind == BIAS_RAY) {
            // the row its ray's warps left in the scratch slot (ordered by the tile barrier of the feature park)
            const float* brow = vb_slot + (q / (p.N >> 5)) * 256;
            wb[0] = __ldcg(reinterpret_cast<const float4*>(brow) + lane);
            wb[1] = __ldcg(reinterpret_cast<const float4*>(brow + 128) + lane);
          } else {
            const long long img = kRender ? (long long)rs.img : s / p.per_image;
            const float* brow = ly.bias_kind == BIAS_RAY ? p.raybias + (s / p.N) * 256 : p.imgbias + img * 256;
            wb[0] = __ldg(reinterpret_cast<const float4*>(brow) + lane);
            wb[1] = __ldg(reinterpret_cast<const float4*>(brow + 128) + lane);
          }
        }
        // Two windows in which both tiles and the tensor pipe wait whatever the epilogue warps do (scripts/fwd_prof.py): right after
        // the feature park the weight stream of the rgb-0 stage queues behind 128 KB of bulk stores in the SM's TMA FIFO
        // (~2 700 cycles), and the trans-0 stage waits for the 64 KB feature reload (~2 100 cycles).  The work that has no place on
        // a tile's critical path goes there: the next super-tile's rays, bounds, jitter and depths (two dependent global
        // loads) into the first, the compositing of the previous super-tile's samples into the second.
        if (kRender && L == kSpillLayer + 1 && st + gridDim.x < n_super) {
          if constexpr (kList) nxt = render_fetch_list(p, (list_shard(p, 0) + st + gridDim.x) * 2 + t, row, lane);
          else nxt = render_fetch(p, (st + gridDim.x) * 2 + t, row, lane);
        }
        if (kRender && L == (kNL > kStaticLayers ? kReloadIssueLayer + 1 : kSpillLayer + 1) && have_done) {
          float* sc = reinterpret_cast<float*>(smem + kOffComp) + t * kCompFloats;      // (the park barrier separates two uses)
          render_composite(p, sc, t, q, lane, done_ray, done_k, done_d, done_dist, done_live, done_v[0], done_v[1], done_v[2], done_v[3],
                           done_v[4], done_v[5], done_v[6], done_v[7], done_v[8]);
          have_done = false;
        }
        if (kRender) {
          // the tile's view-direction bias row is worked out HERE, before the accumulator wait of three consecutive trunk stages
          if (L >= kViewBiasLayer - 2 && L <= kViewBiasLayer) {
            const int wpr = kSmemBias ? 4 : p.N >> 5;      // warps per ray: 4, 2, 1
            float* dst = vb_slot + (q / wpr) * 256;
            if (wpr >= 2) {                // N = 128 / 64: nine inputs per stage
              const int col = (q & (wpr - 1)) * (256 / wpr) + lane * (8 / wpr);
              const int j0 = (L - (kViewBiasLayer - 2)) * 9;
              if (j0 == 0) {
                vb_e = render_view_element(p, rs, lane);
                const float* brow = p.imgbias_rgb + (long long)rs.img * 256 + col;
                vb_acc.x = __ldg(brow); vb_acc.y = __ldg(brow + 1);
                vb_acc.z = wpr == 2 ? __ldg(brow + 2) : 0.f; vb_acc.w = wpr == 2 ? __ldg(brow + 3) : 0.f;
              }
              if (wpr == 4) vb_acc = render_view_batch<2>(p, vb_e, col, j0, vb_acc);
              else vb_acc = render_view_batch<4>(p, vb_e, col, j0, vb_acc);
              if (L == kViewBiasLayer) {
                if (kSmemBias) asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(bias_sm + col * 4), "f"(vb_acc.x), "f"(vb_acc.y) : "memory");
                else if (wpr == 4) *reinterpret_cast<float2*>(dst + col) = make_float2(vb_acc.x, vb_acc.y);
                else *reinterpret_cast<float4*>(dst + col) = vb_acc;
              }
            } else if (L == kViewBiasLayer) {      // N = 32: one warp per ray computes all 256 columns, four at a time
              const float e = render_view_element(p, rs, lane);
              for (int pass = 0; pass < 2; ++pass) {
                const int col = pass * 128 + lane * 4;
                const float* brow = p.imgbias_rgb + (long long)rs.img * 256 + col;
                float4 acc4 = make_float4(__ldg(brow), __ldg(brow + 1), __ldg(brow + 2), __ldg(brow + 3));
                for (int j0 = 0; j0 < 27; j0 += 9) acc4 = render_view_batch<4>(p, e, col, j0, acc4);
                *reinterpret_cast<float4*>(dst + col) = acc4;
              }
            }
          }
        }
        if (!kRender && kMode != 0 && L == kNL - 2 && st + gridDim.x < n_super) {
          // per-sample launches: the same for the next sample's loads (ray, depth) and its sixty sines
          const long long sn_raw = ((st + gridDim.x) * 2 + t) * 128 + row, sn = sn_raw < p.S ? sn_raw : p.S - 1, rn = sn / p.N;
          const float cn[3] = {p.center[rn * 3], p.center[rn * 3 + 1], p.center[rn * 3 + 2]};
          const float dn[3] = {p.ray[rn * 3], p.ray[rn * 3 + 1], p.ray[rn * 3 + 2]};
          encode_regs(cn, dn, p.depth[sn], enc_next);
        }
        mbar_wait(bar_acc(t), acc_ph);
        acc_ph ^= 1;
        tc_fence_after();
        if (ly.epi == EPI_HIDDEN && store_pending) {   // the previous bulk store must have finished reading A_t
          if (row == 0) bulk_wait_read();
          named_bar_sync(1 + t, kTileThreads);
          store_pending = false;
        }
        if (L == kReloadIssueLayer && kNL > kStaticLayers && row == 0) {
          // every MMA that reads A_t has retired (acc barrier) -> bring the trunk feature back for the transient head
          bulk_wait_all();
          fence_proxy_async_all();
          mbar_expect_tx(bar_reload(t), kABytes);
          bulk_g2s(a_smem, p_save ? p_save + ((size_t)(st * 2 + t) * kSaveSlots) * kABytes : my_scratch, kABytes, bar_reload(t));
        }
        if (copy_row) named_bar_sync(1 + t, kTileThreads);      // the tile's 128 threads wrote the row before the accumulator wait
        if (ly.epi == EPI_HIDDEN) {
          const uint32_t a_row = a_smem + row * 16;
          const bool train_stage = p_save && L != kSpillLayer && kSaveSlot[L] >= 0;
          if (train_stage) {
            // training: h1 / h2 of either head also leave a ReLU bitmask [128 rows][256 bits] for the backward chain (word
            // planes [8][128 rows]: plane = 32-column slab, so a warp's store of one slab is 128 contiguous bytes), and the
            // activations go straight from the registers to their saved tile image (the backward's operands): a warp's
            // 16-byte groups cover 512 contiguous bytes and nothing re-reads the A tile
            const int mslot = kMaskBitSlot[L];
            uint32_t* words = mslot < 0 ? nullptr
                                        : reinterpret_cast<uint32_t*>(p.bits + ((size_t)(st * 2 + t) * 4 + mslot) * kMaskBitBytes) + row;
            uint8_t* g_row = p_save + ((size_t)(st * 2 + t) * kSaveSlots + kSaveSlot[L]) * kABytes + row * 16;
            if (ly.bias_kind == BIAS_MMA) {
              hidden_epilogue<false, 8, true>(tmem_row, nullptr, a_row, words, g_row);
            } else if (kSmemBias) {
              hidden_epilogue_sbias<8, true>(tmem_row, bias_sm, a_row, words, g_row);
            } else if (warp_bias) {
              hidden_epilogue_wbias<8, true>(tmem_row, wb, a_row, words, g_row);
            } else {
              const float* bias = ly.bias_kind == BIAS_RAY ? p.raybias + (s / p.N) * 256 : p.imgbias + (s / p.per_image) * 256;
              hidden_epilogue<true, 8, true>(tmem_row, bias, a_row, words, g_row);
            }
          } else if (ly.bias_kind == BIAS_MMA) {
            hidden_epilogue<false, 8>(tmem_row, nullptr, a_row);
          } else if (kSmemBias) {
            hidden_epilogue_sbias<8>(tmem_row, bias_sm, a_row);
          } else if (warp_bias) {
            hidden_epilogue_wbias<8>(tmem_row, wb, a_row);
          } else {
            const float* bias = ly.bias_kind == BIAS_RAY ? p.raybias + (s / p.N) * 256 : p.imgbias + (s / p.per_image) * 256;
            hidden_epilogue<true, 8>(tmem_row, bias, a_row);
          }
          fence_proxy_async_smem();
          if (L == kSpillLayer && kNL > kStaticLayers) {      // static only: no second head, nothing to park
            // park the trunk feature (bf16 tile image) in the L2 scratch (training: in its slot of the save buffer, where
            // the backward also reads it) -- the bulk store overlaps the next stage's MMAs
            named_bar_sync(1 + t, kTileThreads);
            if (row == 0) {
              uint8_t* dst = p_save ? p_save + ((size_t)(st * 2 + t) * kSaveSlots + kSaveSlot[L]) * kABytes : my_scratch;
              bulk_s2g(dst, a_smem, kABytes);
              bulk_commit();
            }
            store_pending = true;
          } else if (kRender && L == kSpillLayer) {
            named_bar_sync(1 + t, kTileThreads);      // static only: nothing is parked, but the view-bias rows need the tile barrier
          }
        } else {
          // N=16 output stage: columns 0..7 = x . bf16(W rows), columns 8..15 = x . bf16(W - bf16(W)) of the same rows
          uint32_t v[16];
          TP_TMEM_LD16(tmem_row, v);
          TP_TMEM_WAIT16(v);
          if (L != kNL - 1) {      // the accumulator is in registers: release the next stage's MMAs before the softplus / sigmoid arithmetic
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_ready(t));
          }
          const float* sb = p.biasbuf + kSmallBiasOffset;
          auto out = [&](int c) { return __uint_as_float(v[c]) + __uint_as_float(v[c + 8]); };
          float rgb_t[3] = {0.f, 0.f, 0.f}, sigma_t = 0.f, unc = 0.f;
          if (ly.epi == EPI_DENSITY) {
            sigma_s = tp_softplus(out(0) + sb[0]);
          } else if (ly.epi == EPI_RGB_OUT) {
#pragma unroll
            for (int c = 0; c < 3; ++c) rgb_s[c] = tp_sigmoid(out(c) + sb[1 + c]);
          } else {
#pragma unroll
            for (int c = 0; c < 3; ++c) rgb_t[c] = tp_sigmoid(out(c) + sb[4 + c]);
            sigma_t = tp_softplus(out(3) + sb[7]);
            unc = tp_softplus(out(4) + sb[8]);
          }
          if (L == kNL - 1) {      // last stage (static only: the rgb output; the transient values stay zero)
            if (kRender) {
              // hand the tile on first: the next super-tile's samples are encoded and its first MMAs released before this
              // one is composited, so the compositing overlaps tensor work instead of leaving the pipe idle
              // the sample is finished: keep its nine values for the compositing (above, next super-tile), encode the next
              // super-tile's sample (its point is known since the rgb-0 stage) and release its first MMAs
              done_ray = rs.ray; done_k = rs.k; done_d = rs.d; done_dist = rs.dist; done_live = rs.live;
              done_v[0] = sigma_s; done_v[1] = sigma_t; done_v[8] = unc;
#pragma unroll
              for (int c = 0; c < 3; ++c) { done_v[2 + c] = rgb_s[c]; done_v[5 + c] = rgb_t[c]; }
              have_done = true;
              if (st + gridDim.x < n_super) {
                rs = nxt;
                render_encode(rs.xyz[0], rs.xyz[1], rs.xyz[2], e_smem, row);
                fence_proxy_async_smem();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_ready(t));
              }
            } else if (live) {
#pragma unroll
              for (int c = 0; c < 3; ++c) *reinterpret_cast<float2*>(p.rgb + s * 6 + c * 2) = make_float2(rgb_s[c], rgb_t[c]);
              *reinterpret_cast<float2*>(p.density + s * 2) = make_float2(sigma_s, sigma_t);
              p.uncert[s] = unc;
            }
          }
        }
        if (L != kNL - 1 && !ly.small) {   // (output stages arrived above; the next super-tile's encode covers the last stage)
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_ready(t));
        }
      }
    }
    if (kRender && have_done) {      // the last super-tile of this CTA
      float* sc = reinterpret_cast<float*>(smem + kOffComp) + t * kCompFloats;
      render_composite(p, sc, t, q, lane, done_ray, done_k, done_d, done_dist, done_live, done_v[0], done_v[1], done_v[2], done_v[3],
                       done_v[4], done_v[5], done_v[6], done_v[7], done_v[8]);
    }
    if (row == 0) bulk_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ------------------------------------------------------------------------------------------ helper kernels

// desc row: [w_ptr, ld, row0, rows_valid, col0, cols_valid, n_layout, bias_ptr, bias_klocal, transpose]
// transpose != 0: chunk element (n, kl) = W[col0 + kl][row0 + n]  (B operand of the input-gradient GEMMs, dX = dZ W)
// (bias_ptr != 0: element (n, bias_klocal) of the chunk is bias[n] -- the column multiplied by the constant-1 of E)
__global__ void pack_weights_kernel(const long long* __restrict__ desc, __nv_bfloat16* __restrict__ out) {
  const long long* d = desc + (long long)blockIdx.x * 10;
  const float* W = reinterpret_cast<const float*>(d[0]);
  const long long ld = d[1], row0 = d[2], rows_valid = d[3], col0 = d[4], cols_valid = d[5], n_layout = d[6];
  const float* bias = reinterpret_cast<const float*>(d[7]);
  const long long bias_k = d[8], transpose = d[9];
  __nv_bfloat16* o = out + (long long)blockIdx.x * (kChunkBytes / 2);
  for (int e = threadIdx.x; e < (int)(kChunkBytes / 2); e += blockDim.x) {
    int n, kl;
    bool in_layout = true;
    if (n_layout == 256) {
      kl = (e >> 11) * 8 + (e & 7);
      n = (e >> 3) & 255;
    } else {
      kl = (e >> 7) * 8 + (e & 7);
      n = (e >> 3) & 15;
      in_layout = e < 4096;
    }
    // N=16 output chunks carry every weight row twice: rows 0..7 = bf16(W), rows 8..15 = bf16(W - bf16(W)) (the epilogue
    // adds accumulator columns c and c + 8)
    const bool lo_part = n_layout == 16 && n >= 8;
    if (n_layout == 16) n &= 7;
    float v = 0.f;
    if (in_layout && W && n < rows_valid && kl < cols_valid)
      v = transpose ? W[(col0 + kl) * ld + row0 + n] : W[(row0 + n) * ld + col0 + kl];
    if (in_layout && bias && kl == bias_k && n < rows_valid) v = bias[n];
    if (lo_part) v -= __bfloat162float(__float2bfloat16_rn(v));
    o[e] = __float2bfloat16_rn(v);
  }
}

// out[b, n] = bias[n] + sum_j W[n, col0 + j] * latent[b, j] for both heads in one launch: blocks [0, B) the rgb head's rows,
// [B, 2B) the transient head's
__global__ void image_biases_kernel(const float* __restrict__ W_r, long long ld_r, int col_r, int n_r, const float* __restrict__ b_r,
                                    const float* __restrict__ lat_r, const float* __restrict__ W_t, long long ld_t, int col_t, int n_t,
                                    const float* __restrict__ b_t, const float* __restrict__ lat_t, int B, float* __restrict__ out_r,
                                    float* __restrict__ out_t) {
  const bool second = (int)blockIdx.x >= B;
  const int b = second ? blockIdx.x - B : blockIdx.x;
  const float* W = second ? W_t : W_r;
  const long long ldw = second ? ld_t : ld_r;
  const int col0 = second ? col_t : col_r, ncols = second ? n_t : n_r;
  const float* bias = second ? b_t : b_r;
  const float* latent = second ? lat_t : lat_r;
  float* out = second ? out_t : out_r;
  const int n = threadIdx.x;
  float acc = bias ? bias[n] : 0.f;
  for (int j = 0; j < ncols; ++j) acc = fmaf(W[n * ldw + col0 + j], latent[(long long)b * ncols + j], acc);
  out[(long long)b * 256 + n] = acc;
}

// out[r, n] = imgbias[r / rays_per_image, n] + sum_j W[n, col0 + j] * viewenc(r)[j];  viewenc = [u, enc(u)], u = ray/|ray|.
// Thread n keeps its weight row in registers; a CTA strides over groups of kRaysPerBlock rays: all encodings of the group first
// (one thread per ray and coordinate), then every thread streams the group's rays; stores are 1 KB-coalesced rows.
constexpr int kRaysPerBlock = 64;
__global__ void __launch_bounds__(256) ray_bias_kernel(const float* __restrict__ ray, long long R, long long rays_per_image,
                                                       int L, const float* __restrict__ W, long long ldw, int col0,
                                                       const float* __restrict__ imgbias, float* __restrict__ out) {
  __shared__ __align__(16) float enc[kRaysPerBlock][28];      // rows of 7 float4: the inner product reads them as broadcast LDS.128
  const int vc = 3 + 6 * L;     // <= 27 (L_view <= 4)
  // the thread's weight row (27 strided, uncoalesced loads) is fetched ONCE: the CTA then strides over groups of rays
  float w[27];
  const int n = threadIdx.x;
#pragma unroll
  for (int j = 0; j < 27; ++j) w[j] = j < vc ? W[n * ldw + col0 + j] : 0.f;
  const long long n_groups = (R + kRaysPerBlock - 1) / kRaysPerBlock;
  for (long long grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
    const long long r0 = grp * kRaysPerBlock;
    __syncthreads();      // the previous group's encodings are no longer read
    if (threadIdx.x < kRaysPerBlock * 3) {      // one thread per (ray, coordinate): unit component, then its 2L encodings
      const int rr = threadIdx.x / 3, cc = threadIdx.x - rr * 3;
      const long long r = r0 + rr;
      const bool live = r < R;
      float uc = 0.f;
      if (live) {
        const float x = ray[r * 3], y = ray[r * 3 + 1], z = ray[r * 3 + 2];
        uc = __fdiv_rn(cc == 0 ? x : (cc == 1 ? y : z), unit_length(x, y, z));      // same bits as the render launch's in-kernel row
      }
      enc[rr][cc] = uc;
      for (int k = 0; k < L; ++k) {
        const float arg = __fmul_rn(uc, ldexpf(3.14159265358979323846f, k));
        enc[rr][3 + cc * 2 * L + k] = live ? sinf(arg) : 0.f;
        enc[rr][3 + cc * 2 * L + L + k] = live ? cosf(arg) : 0.f;
      }
    } else {      // the other threads clear the pad columns (vc .. 27)
      for (int i = threadIdx.x - kRaysPerBlock * 3; i < kRaysPerBlock * (28 - vc); i += blockDim.x - kRaysPerBlock * 3)
        enc[i / (28 - vc)][vc + i % (28 - vc)] = 0.f;
    }
    __syncthreads();
    // four rays per iteration: four independent fma chains per thread (the 27-long chain of one ray is latency-bound)
    const long long img_first = r0 / rays_per_image;
    for (int rr = 0; rr < kRaysPerBlock; rr += 4) {
      float acc[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const long long r = r0 + rr + q;
        long long img = img_first;
        while (r >= (img + 1) * rays_per_image) ++img;
        acc[q] = r < R ? imgbias[img * 256 + n] : 0.f;
      }
#pragma unroll
      for (int j4 = 0; j4 < 7; ++j4) {      // per ray the same fma order as column by column (the pad column is skipped)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 e = reinterpret_cast<const float4*>(enc[rr + q])[j4];
          acc[q] = fmaf(w[4 * j4], e.x, acc[q]);
          acc[q] = fmaf(w[4 * j4 + 1], e.y, acc[q]);
          acc[q] = fmaf(w[4 * j4 + 2], e.z, acc[q]);
          if (j4 < 6) acc[q] = fmaf(w[4 * j4 + 3], e.w, acc[q]);
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (r0 + rr + q < R) __stcs(out + (r0 + rr + q) * 256 + n, acc[q]);      // 315 MB per frame, read once by the fused kernel
    }
  }
}

}  // namespace tc

TP_API int tp_tc_num_chunks(void) { return tc::kNumChunks; }
TP_API int64_t tp_tc_chunk_bytes(void) { return tc::kChunkBytes; }
// parked features (2 x 64 KB per CTA) + view-bias rows of the render launch (2 tiles x 4 rays x 1 KB per CTA) + the cycle
// counters of a -DTP_FWD_PROF build (scripts/fwd_prof.py; [CTA][tile][stage][4] int64, untouched otherwise)
TP_API int64_t tp_tc_scratch_bytes(void) { return (int64_t)tp_num_sms() * (2 * tc::kABytes + 2 * 4 * 1024 + 2 * tc::kNumLayers * 4 * 8); }
TP_API int64_t tp_tc_prof_offset(void) { return (int64_t)tp_num_sms() * (2 * tc::kABytes + 2 * 4 * 1024); }

// save buffer: [tiles][7][64 KB] tile images, then [tiles][4][4 KB] ReLU bitmasks (tiles rounded up to whole super-tiles)
TP_API int64_t tp_tc_save_bytes(int64_t S) {
  return ((S + 255) / 256) * 2 * (tc::kSaveSlots * (int64_t)tc::kABytes + tc::kMaskBitSlots * (int64_t)tc::kMaskBitBytes);
}

TP_API int tp_tc_pack_weights(const int64_t* chunk_desc, int n_chunks, void* packed, void* stream) {
  if (!chunk_desc || !packed) return TP_ERR_BAD_ARG;
  if (n_chunks < 1) return TP_ERR_BAD_SHAPE;
  tc::pack_weights_kernel<<<n_chunks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const long long*>(chunk_desc),
                                                                    reinterpret_cast<__nv_bfloat16*>(packed));
  return tp_launch_status();
}

TP_API int tp_tc_image_biases(const float* W_rgb, int64_t ld_rgb, int col_rgb, int n_light, const float* b_rgb, const float* light,
                              const float* W_trans, int64_t ld_trans, int col_trans, int n_trans, const float* b_trans,
                              const float* trans, int B, float* out_rgb, float* out_trans, void* stream) {
  if (!W_rgb || !light || !out_rgb || !W_trans || !trans || !out_trans) return TP_ERR_BAD_ARG;
  if (B < 1 || n_light < 0 || n_trans < 0) return TP_ERR_BAD_SHAPE;
  tc::image_biases_kernel<<<2 * B, 256, 0, (cudaStream_t)stream>>>(W_rgb, ld_rgb, col_rgb, n_light, b_rgb, light, W_trans, ld_trans,
                                                                col_trans, n_trans, b_trans, trans, B, out_rgb, out_trans);
  return tp_launch_status();
}

TP_API int tp_tc_ray_bias(const float* ray, int64_t R, int64_t rays_per_image, int L_view, const float* W, int64_t ldw,
                          int col0, const float* imgbias, float* out, void* stream) {
  if (!ray || !W || !imgbias || !out) return TP_ERR_BAD_ARG;
  if (R < 0 || rays_per_image < 1 || L_view < 0 || L_view > 4) return TP_ERR_BAD_SHAPE;
  if (R == 0) return TP_OK;
  const long long n_groups = (R + tc::kRaysPerBlock - 1) / tc::kRaysPerBlock, cap = (long long)tp_num_sms() * 6;
  tc::ray_bias_kernel<<<(unsigned)(n_groups < cap ? n_groups : cap), 256, 0, (cudaStream_t)stream>>>(
      ray, R, rays_per_image, L_view, W, ldw, col0, imgbias, out);
  return tp_launch_status();
}

// 8 epilogue warps drain the accumulators (256 columns per thread, 320 threads per CTA): the same tensor-pipe time as 16 warps,
// but the narrower CTA draws less power and the capped clock settles higher -- 2 % faster for the C2 frame, 1.7 % for the C3
// training step (same-box A/B, profiles/r01f_summary.md section 9).
static int tc_launch(void (*kern)(const tc::Params), const tc::Params& p, int grid, cudaStream_t stream) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::kSmemBytes);
  if (e != cudaSuccess) return (int)e;
  kern<<<grid, tc::kThreads, tc::kSmemBytes, stream>>>(p);
  return tp_launch_status();
}

TP_API int tp_tc_nerf_stl_forward(const float* center, const float* ray, const float* depth, int64_t S, int N,
                                  int64_t per_image, const void* packed, const float* biasbuf, const float* raybias,
                                  const float* imgbias, float* rgb, float* density, float* uncert, void* scratch,
                                  int64_t scratch_bytes, void* save, int flags, void* stream) {
  if (!center || !ray || !depth || !packed || !biasbuf || !raybias || !imgbias || !rgb || !density || !uncert || !scratch)
    return TP_ERR_BAD_ARG;
  if (S < 0 || N < 1 || per_image < 1) return TP_ERR_BAD_SHAPE;
  if (((uintptr_t)packed & 15) || ((uintptr_t)scratch & 15) || ((uintptr_t)biasbuf & 15) || ((uintptr_t)raybias & 15) ||
      ((uintptr_t)imgbias & 15) || ((uintptr_t)rgb & 7) || ((uintptr_t)density & 7) || ((uintptr_t)save & 15))
    return TP_ERR_ALIGN;
  if (flags & ~(1 << 17)) return TP_ERR_BAD_ARG;
  if (!tp_device_is_sm100()) return TP_ERR_ARCH;
  if (S == 0) return TP_OK;
  const long long n_super = (S + 255) / 256;
  int grid = tp_num_sms();
  if (n_super < grid) grid = (int)n_super;
  if (scratch_bytes < (int64_t)grid * 2 * tc::kABytes) return TP_ERR_WORKSPACE;
  tc::Params p = {};
  p.center = center; p.ray = ray; p.depth = depth; p.S = S; p.N = N; p.per_image = per_image;
  p.packed = reinterpret_cast<const uint8_t*>(packed); p.biasbuf = biasbuf; p.raybias = raybias; p.imgbias = imgbias;
  p.rgb = rgb; p.density = density; p.uncert = uncert; p.scratch = reinterpret_cast<uint8_t*>(scratch);
  p.save = reinterpret_cast<uint8_t*>(save);
  p.bits = save ? p.save + ((S + 255) / 256) * 2 * tc::kSaveSlots * (size_t)tc::kABytes : nullptr;
  p.prof_offset = tp_tc_prof_offset();
  p.n_layers = (flags & (1 << 17)) ? tc::kStaticLayers : tc::kNumLayers;      // flags bit 17: static-only rendering
  if ((flags & (1 << 17)) && save) return TP_ERR_BAD_ARG;                     // inference launches only
  const bool stat = p.n_layers == tc::kStaticLayers;
  const bool n128 = N == 128;      // one ray (and one image) per tile: bias rows in shared memory
  void (*kern)(const tc::Params) =
      N % 32 != 0 ? (stat ? tc::nerf_stl_forward_kernel<tc::kStaticLayers> : tc::nerf_stl_forward_kernel<tc::kNumLayers>)
      : !save     ? (stat ? (n128 ? tc::nerf_stl_forward_kernel<tc::kStaticLayers, 1, true> : tc::nerf_stl_forward_kernel<tc::kStaticLayers, 1>)
                          : (n128 ? tc::nerf_stl_forward_kernel<tc::kNumLayers, 1, true> : tc::nerf_stl_forward_kernel<tc::kNumLayers, 1>))
                  : (n128 ? tc::nerf_stl_forward_kernel<tc::kNumLayers, 2, true> : tc::nerf_stl_forward_kernel<tc::kNumLayers, 2>);
  return tc_launch(kern, p, grid, (cudaStream_t)stream);
}

// Graph.render after ray selection (model/nerf_adapt_st_gan.py:565-631) as ONE launch.
TP_API int tp_render_fused_forward(const float* kinv, const float* pose_inv, int B, int H, int W, float pix_offset,
                                   const int64_t* ray_idx, int64_t R, int64_t ray0, const float* z_near, const float* z_far,
                                   int N, int depth_mode, const float* rand, uint64_t seed, const void* packed,
                                   const float* biasbuf, const float* wview, int L_view, const float* imgbias_rgb,
                                   const float* imgbias_trans, float min_uncert, float* rgb, float* rgb_static,
                                   float* rgb_transient, float* depth, float* opacity, float* opacity_static,
                                   float* opacity_transient, float* uncert, float* alpha_static, float* alpha_transient,
                                   float* density, void* scratch, int64_t scratch_bytes, int flags, void* stream) {
  if (!kinv || !pose_inv || !z_near || !z_far || !packed || !biasbuf || !wview || !imgbias_rgb || !imgbias_trans || !scratch)
    return TP_ERR_BAD_ARG;
  if (B < 1 || H < 1 || W < 1 || R < 0 || L_view < 0 || L_view > 4) return TP_ERR_BAD_SHAPE;
  if (N != 32 && N != 64 && N != 128) return TP_ERR_BAD_SHAPE;      // a 128-row tile holds whole rays
  if (depth_mode < 0 || depth_mode > 2 || (depth_mode == 0 && !rand)) return TP_ERR_BAD_ARG;
  if (!ray_idx && (ray0 < 0 || ray0 + R > (int64_t)H * W)) return TP_ERR_BAD_SHAPE;
  if (flags & ~(1 << 17)) return TP_ERR_BAD_ARG;
  if (((uintptr_t)packed & 15) || ((uintptr_t)scratch & 15) || ((uintptr_t)wview & 15) || ((uintptr_t)imgbias_rgb & 15) ||
      ((uintptr_t)imgbias_trans & 15) || ((uintptr_t)density & 7))
    return TP_ERR_ALIGN;
  if (!tp_device_is_sm100()) return TP_ERR_ARCH;
  const int64_t S = (int64_t)B * R * N;
  if (S == 0) return TP_OK;
  const long long n_super = (S + 255) / 256;
  int grid = tp_num_sms();
  if (n_super < grid) grid = (int)n_super;
  if (scratch_bytes < (int64_t)grid * (2 * tc::kABytes + 2 * 4 * 1024)) return TP_ERR_WORKSPACE;
  tc::Params p = {};
  p.S = S; p.N = N; p.per_image = R * N;
  p.packed = reinterpret_cast<const uint8_t*>(packed); p.biasbuf = biasbuf; p.imgbias = imgbias_trans;
  p.density = density; p.scratch = reinterpret_cast<uint8_t*>(scratch);
  p.prof_offset = tp_tc_prof_offset();
  p.n_layers = (flags & (1 << 17)) ? tc::kStaticLayers : tc::kNumLayers;
  p.kinv = kinv; p.pinv = pose_inv; p.H = H; p.W = W; p.pix_offset = pix_offset;
  p.ray_idx = reinterpret_cast<const long long*>(ray_idx); p.R = R; p.ray0 = ray0;
  p.z_near = z_near; p.z_far = z_far; p.rand = rand; p.depth_mode = depth_mode; p.seed = seed;
  p.wview = wview; p.L_view = L_view; p.imgbias_rgb = imgbias_rgb; p.min_uncert = min_uncert;
  p.o_rgb = rgb; p.o_rgb_s = rgb_static; p.o_rgb_t = rgb_transient; p.o_depth = depth; p.o_op = opacity;
  p.o_op_s = opacity_static; p.o_op_t = opacity_transient; p.o_unc = uncert; p.o_as = alpha_static; p.o_at = alpha_transient;
  const bool stat = p.n_layers == tc::kStaticLayers, n128 = N == 128;
  void (*kern)(const tc::Params) =
      stat ? (n128 ? tc::nerf_stl_forward_kernel<tc::kStaticLayers, 3, true> : tc::nerf_stl_forward_kernel<tc::kStaticLayers, 3>)
           : (n128 ? tc::nerf_stl_forward_kernel<tc::kNumLayers, 3, true> : tc::nerf_stl_forward_kernel<tc::kNumLayers, 3>);
  return tc_launch(kern, p, grid, (cudaStream_t)stream);
}

// The same launch over an object-pixel list (kMode 4): one CTA per SM, since the host does not know the list's length; rank
// shard_rank of shard_world renders its share of the list's super-tiles.
TP_API int tp_render_fused_forward_list(const float* kinv, const float* pose_inv, int B, int H, int W, float pix_offset,
                                        const int64_t* list, const int64_t* n_slots, int shard_rank, int shard_world,
                                        const float* z_near, const float* z_far, int N, int depth_mode, const float* rand,
                                        uint64_t seed, const void* packed, const float* biasbuf, const float* wview, int L_view,
                                        const float* imgbias_rgb, const float* imgbias_trans, float min_uncert, float* rgb,
                                        float* rgb_static, float* rgb_transient, float* depth, float* opacity,
                                        float* opacity_static, float* opacity_transient, float* uncert, float* alpha_static,
                                        float* alpha_transient, float* density, void* scratch, int64_t scratch_bytes, int flags,
                                        void* stream) {
  if (!kinv || !pose_inv || !list || !n_slots || !z_near || !z_far || !packed || !biasbuf || !wview || !imgbias_rgb ||
      !imgbias_trans || !scratch)
    return TP_ERR_BAD_ARG;
  if (B < 1 || H < 1 || W < 1 || L_view < 0 || L_view > 4) return TP_ERR_BAD_SHAPE;
  if (N != 32 && N != 64 && N != 128) return TP_ERR_BAD_SHAPE;
  if (depth_mode < 0 || depth_mode > 2 || (depth_mode == 0 && !rand)) return TP_ERR_BAD_ARG;      // rand: [B*H*W*N], frame-sized
  if (shard_world < 1 || shard_rank < 0 || shard_rank >= shard_world) return TP_ERR_BAD_ARG;
  if (flags & ~(1 << 17)) return TP_ERR_BAD_ARG;
  if (((uintptr_t)packed & 15) || ((uintptr_t)scratch & 15) || ((uintptr_t)wview & 15) || ((uintptr_t)imgbias_rgb & 15) ||
      ((uintptr_t)imgbias_trans & 15) || ((uintptr_t)density & 7))
    return TP_ERR_ALIGN;
  if (!tp_device_is_sm100()) return TP_ERR_ARCH;
  const int grid = tp_num_sms();
  if (scratch_bytes < (int64_t)grid * (2 * tc::kABytes + 2 * 4 * 1024)) return TP_ERR_WORKSPACE;
  tc::Params p = {};
  p.S = 0; p.N = N; p.per_image = (int64_t)H * W * N;      // (list mode takes its rays and its length from the list)
  p.list = reinterpret_cast<const long long*>(list); p.n_slots = reinterpret_cast<const long long*>(n_slots);
  p.shard_rank = shard_rank; p.shard_world = shard_world;
  p.packed = reinterpret_cast<const uint8_t*>(packed); p.biasbuf = biasbuf; p.imgbias = imgbias_trans;
  p.density = density; p.scratch = reinterpret_cast<uint8_t*>(scratch);
  p.prof_offset = tp_tc_prof_offset();
  p.n_layers = (flags & (1 << 17)) ? tc::kStaticLayers : tc::kNumLayers;
  p.kinv = kinv; p.pinv = pose_inv; p.H = H; p.W = W; p.pix_offset = pix_offset;
  p.z_near = z_near; p.z_far = z_far; p.rand = rand; p.depth_mode = depth_mode; p.seed = seed;
  p.wview = wview; p.L_view = L_view; p.imgbias_rgb = imgbias_rgb; p.min_uncert = min_uncert;
  p.o_rgb = rgb; p.o_rgb_s = rgb_static; p.o_rgb_t = rgb_transient; p.o_depth = depth; p.o_op = opacity;
  p.o_op_s = opacity_static; p.o_op_t = opacity_transient; p.o_unc = uncert; p.o_as = alpha_static; p.o_at = alpha_transient;
  const bool stat = p.n_layers == tc::kStaticLayers, n128 = N == 128;
  void (*kern)(const tc::Params) =
      stat ? (n128 ? tc::nerf_stl_forward_kernel<tc::kStaticLayers, 4, true> : tc::nerf_stl_forward_kernel<tc::kStaticLayers, 4>)
           : (n128 ? tc::nerf_stl_forward_kernel<tc::kNumLayers, 4, true> : tc::nerf_stl_forward_kernel<tc::kNumLayers, 4>);
  return tc_launch(kern, p, grid, (cudaStream_t)stream);
}
