// K2 (fp32-parity mode on the tensor cores): fused per-sample NeRF forward with SPLIT-bf16 operands, sm_100a.
//
// The <= 1e-4 contract of NeRF.forward (layers/nerf_static_transient_light.py:76-145, layers/nerf.py:61-99) needs ~16
// mantissa bits per operand; bf16 has 8.  Every operand therefore exists twice -- x = hi + lo with hi = bf16(x),
// lo = bf16(x - hi) -- and every K = 16 step is three tcgen05.mma passes into one fp32 TMEM accumulator:
//
//        D += A_hi W_hi^T  +  A_hi W_lo^T  +  A_lo W_hi^T            (the dropped A_lo W_lo^T term is 2^-18 relative)
//
// so the fp32 parity mode runs at a third of the bf16 tensor rate instead of at SIMT FFMA rate (mlp_simt.cu).
//
// Work decomposition (one persistent 320-thread CTA per SM, one 128-sample tile at a time):
//   * activations live in SMEM as two tile images (A_hi, A_lo: [32 k8][128 rows][8] bf16, K-major core-matrix layout), the
//     fp32 positional encoding (reference bits: sin(fl(x * fl(2^k pi)))) as E_hi, E_lo; nothing but the parked trunk feature
//     and the per-sample outputs ever leaves the SM;
//   * weights stream through a 4-slot ring of 16 KB slots, one slot per K = 16 step: [W_hi 8 KB | W_lo 8 KB], each
//     [2 k8][256 rows][8]; the N = 16 output stages stream one 8 KB slot [32 k8][16 rows][8] whose rows 0..7 hold W_hi and
//     rows 8..15 W_lo (two passes, A_hi and A_lo; the epilogue adds accumulator columns c and c + 8);
//   * BOTH 256-column TMEM accumulators are used by ONE tile, alternating by stage, and the drain of stage L publishes the next
//     A operand in eight 32-column groups (one mbarrier each): the MMAs of stage L+1 start as soon as the first group is
//     written and overlap the rest of the drain -- the tensor pipe only idles for the first slab of every drain;
//   * biases are added in fp32 by the drain (static vectors, the per-ray row of tp_tc_ray_bias, the per-image row of
//     tp_tc_image_biases): no bf16 rounding of any bias;
//   * the stage list is DATA (tp_tc32_forward's `stages`): trunk depth, skip positions and head depths come from the caller's
//     architecture, not from a table compiled into the kernel.
//
// Render launch (tp_tc32_render_forward, either arithmetic): the tile's rows make their own samples from the pixel index (rays,
// bounds, jitter, depths: the bits of tp_raygen + tp_sample_depth), the rgb-0 stage's per-ray bias row is computed by the warps
// that read it (tp_tc_ray_bias's bits, in a per-warp slot of the L2-resident scratch), and the last stage's samples are
// composited in the epilogue (row = sample: warp scan + cross-warp carry) -- no per-sample tensor and no bias table in HBM.
//
// SMEM: A_hi 64K | A_lo 64K | E_hi 16K | E_lo 16K | ring 4 x 16K | barriers = 229 632 B (+ 512 B compositing scratch in the
// render launch).  TMEM: 512 columns.
#include <type_traits>
#include <cuda_fp16.h>
#include "tc_common.cuh"
#include "rays.cuh"
#include "../../include/texpose_b200.h"

namespace tcs {
using namespace tc;

constexpr int kThreads = 320;                  // warps 0-7 drain / encode, warp 8 weight producer, warp 9 MMA issuer
constexpr int kProducerWarp = 8, kMmaWarp = 9;
constexpr int kRing = 4;
constexpr uint32_t kSlotBytes = 16384, kHalfSlot = 8192;
constexpr uint32_t kEBytes = 16384;            // 128 x 64 bf16
constexpr uint32_t kOffAhi = 0, kOffAlo = kABytes, kOffEhi = 2 * kABytes, kOffElo = kOffEhi + kEBytes;
constexpr uint32_t kOffRing = kOffElo + kEBytes;
constexpr uint32_t kOffBar = kOffRing + kRing * kSlotBytes;
constexpr uint32_t kSmemBytes = kOffBar + 256;
static_assert(kSmemBytes <= 232448, "227 KB of shared memory per CTA");
constexpr int kMaxStages = 24;
constexpr int kEncL = 10;                      // frequencies of the point encoding (the reference's yaml files: L_3D = 10)

enum Kind : int { KIND_HIDDEN = 0, KIND_DENSITY = 1, KIND_RGB_OUT = 2, KIND_TRANS_OUT = 3 };
enum BiasKind : int { BIAS_STATIC = 0, BIAS_RAY = 1, BIAS_IMAGE = 2 };
enum Flags : int {
  F_WAIT_READY = 1,    // the stage reads the A operand the previous hidden stage's drain writes
  F_RELOAD = 2,        // the stage reads the parked trunk feature (bulk-loaded back into A)
  F_PARK = 4,          // the stage's output is the trunk feature: the drain also stores it to the CTA's scratch
  F_E_LAST = 8         // last stage of the tile that reads E: the next tile's encoding may be written once its MMAs retired
};
struct Stage {
  int a_steps, e_steps, kind, bias_kind, bias_off, flags, save_slot;      // save_slot: -1, or the tile-image slot the stage's output is kept in
};
struct Params {
  const float* center;       // [rays,3]
  const float* ray;          // [rays,3]
  const float* depth;        // [S]
  long long S;
  int N;
  long long per_image;
  const uint8_t* image;      // weight slots in consumption order (n_slots x 16 KB)
  const float* bias;         // static biases (fp32), addressed by Stage::bias_off
  const float* raybias;      // [rays,256]
  const float* imgbias;      // [images,256]
  float* rgb;                // [S,3,2]
  float* density;            // [S,2]
  float* uncert;             // [S]
  uint8_t* scratch;          // gridDim.x x 128 KB (parked feature, hi | lo), then one 32-bit status word
  unsigned int* status;      // bit 0 is set when a hidden activation left the fp16 range of the split mode (the launch's results are
                             // then not the <= 1e-4 ones): read back by the caller off the hot path (mlp_tc32.check_range)
  uint8_t* save;             // single-pass mode, training: [tiles][n_save][64 KB] bf16 tile images of the stages with a save slot
  int n_save;
  uint32_t* save_bits;       // behind the images: [tiles][n_save][8 planes][128 rows] ReLU bitmasks (plane = 32-column slab, bit = column
                             // is positive): what the backward chain masks with instead of re-reading the 64 KB tiles
  int enc_slot;              // -1, or the save slot that receives the encoding tile [x, enc(x), 1] (zero beyond column 63): the B
                             // operand of the weight-gradient GEMMs of the layers that read the encoding (column 63 = 1: their bias sums)
  int n_stages;
  Stage st[kMaxStages];
};

// The render launch's parameters: the staged kernel's, minus the per-sample inputs / outputs (center, ray, depth, raybias, rgb,
// density, uncert stay unused), plus what a row needs to make its sample and what the compositing writes.
constexpr uint32_t kOffComp = kSmemBytes;                 // [4 warps][3] scan totals, then [4 warps][14] per-ray partial sums
constexpr uint32_t kSmemRender = kOffComp + 512;
static_assert(kSmemRender <= 232448, "227 KB of shared memory per CTA");
constexpr int kViewRowFloats = 128;                       // per drain warp: its column half of the ray's rgb-0 bias row
struct RenderParams : Params {
  const float* kinv;         // [B,9]
  const float* pinv;         // [B,12]
  int H, W;
  float pix_offset;
  const long long* ray_idx;  // [B,R] pixel indices, or NULL: ray r of every view is pixel ray0 + r
  long long R, ray0;
  const float* z_near;       // [B,H*W]
  const float* z_far;
  int depth_mode;            // 0 injected rand [B*R*N], 1 midpoints, 2 Philox (tp_sample_depth's stream)
  const float* rand;
  unsigned long long seed;
  const float* wview;        // [3+6L,256]: the view-encoding columns of the rgb-0 layer, transposed
  int L_view;
  const float* imgbias_rgb;  // [B,256]
  int chains;                // 1: plain model (per-sample density is [S]); 3: static / transient / light ([S,2])
  float min_uncert;
  float *o_rgb, *o_rgb_s, *o_rgb_t, *o_depth, *o_op, *o_op_s, *o_op_t, *o_unc, *o_as, *o_at, *o_density;
  long long vrow_off;        // byte offset in scratch of the view-bias rows: [CTA][8 drain warps][128] floats
};
// The render launch over an object-pixel list (tp_tc32_render_forward_list): ray j of the launch is slot j of the list
// (tp_mask_ray_list), entry q = view * HW + pixel, a pad entry ~(view * HW) is pixel 0 of its view and stores nothing.  Its rays,
// jitter keys and output addresses are those of pixel q of a full-frame launch (ray_idx NULL, ray0 = 0, R = HW).
struct ListRenderParams : RenderParams {
  const long long* list;
  const long long* n_slots;  // device: list entries, a multiple of 256 / N (whole super-tiles = two 128-row tiles, one view each)
  int shard_rank, shard_world;      // this rank renders super-tiles [floor(r T / w), floor((r + 1) T / w)), T = n_slots N / 256
};

// hi / lo fp16 words of two fp32 values (x0 in the low half): hi = fp16(x), lo = fp16(x - hi) -> x to ~22 mantissa bits
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ void split2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  hi = pack_f16(x0, x1);
  const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&hi));
  lo = pack_f16(x0 - h.x, x1 - h.y);
}
// instruction descriptor, kind::f16 with FP16 operands (format fields 0), fp32 accumulate, both K-major
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void umma3(uint32_t d, uint32_t ah, uint32_t al, uint32_t a_hi, uint32_t bh, uint32_t bl, uint32_t b_hi,
                                      uint32_t idesc, uint32_t acc) {
  umma_bf16_lohi(d, ah, a_hi, bh, b_hi, idesc, acc);
  umma_bf16_lohi(d, ah, a_hi, bl, b_hi, idesc, 1u);
  umma_bf16_lohi(d, al, a_hi, bh, b_hi, idesc, 1u);
}

// ------------------------------------------------------------------------------------------ render pieces
// One row's sample: ray from the pixel index (camera.py:292-314, unproject = tp_raygen's arithmetic), depth from the ray's bounds
// (model/nerf_adapt_st_gan.py:682-700, tp_sample_depth's arithmetic and Philox stream), the interval to the next sample of the
// ray and the point.  Rows past the last ray take the last ray (a tile holds whole rays: they are never composited into output).
struct RenderSample {
  long long ray;
  int k;
  bool live;
  float d, dist, xyz[3];
};

__device__ __forceinline__ long long render_ray(const RenderParams& p, long long tile, int row, bool& live) {
  const long long n_rays = p.S / p.N, ray_raw = tile * (128 / p.N) + row / p.N;
  live = ray_raw < n_rays;
  return live ? ray_raw : n_rays - 1;
}
__device__ __forceinline__ void render_unproject(const RenderParams& p, long long ray, long long& b, long long& pix, float c[3],
                                                 float dir[3]) {
  b = ray / p.R;
  pix = p.ray_idx ? p.ray_idx[ray] : p.ray0 + (ray - b * p.R);
  unproject(p.kinv + b * 9, p.pinv + b * 12, __fadd_rn((float)(pix % p.W), p.pix_offset), __fadd_rn((float)(pix / p.W), p.pix_offset),
            c, dir);
}
// first (end = 0) / one past the last (end = 1) 128-row tile of this rank's share of the list
__device__ __forceinline__ long long list_tiles(const ListRenderParams& p, int end) {
  return 2 * (*p.n_slots / (256 / p.N) * (p.shard_rank + end) / p.shard_world);
}
// tiles of the launch; list mode: of this rank's share of the list (render_ray adds the first one's index)
template <class P>
__device__ __forceinline__ long long launch_tiles(const P& p) { return (p.S + 127) / 128; }
__device__ __forceinline__ long long launch_tiles(const ListRenderParams& p) { return list_tiles(p, 1) - list_tiles(p, 0); }
// view of a row (the per-image bias row it reads): its sample's; list mode: its list entry's
template <class P>
__device__ __forceinline__ long long image_of(const P& p, long long tile, int row, long long s) { return s / p.per_image; }
__device__ __forceinline__ long long image_of(const ListRenderParams& p, long long tile, int row, long long s);
// list mode: the "ray" of a row is its frame position q (a pad: pixel 0 of its view, not live)
__device__ __forceinline__ long long render_ray(const ListRenderParams& p, long long tile, int row, bool& live) {
  const long long q = p.list[(list_tiles(p, 0) + tile) * (128 / p.N) + row / p.N];
  live = q >= 0;
  return live ? q : ~q;
}
__device__ __forceinline__ long long image_of(const ListRenderParams& p, long long tile, int row, long long s) {
  bool live;
  return render_ray(p, tile, row, live) / ((long long)p.H * p.W);
}
__device__ __forceinline__ void render_unproject(const ListRenderParams& p, long long ray, long long& b, long long& pix, float c[3],
                                                 float dir[3]) {
  const long long HW = (long long)p.H * p.W;
  b = ray / HW;
  pix = ray - b * HW;
  unproject(p.kinv + b * 9, p.pinv + b * 12, __fadd_rn((float)(pix % p.W), p.pix_offset), __fadd_rn((float)(pix / p.W), p.pix_offset),
            c, dir);
}

// jitter of this lane's sample and of the next sample of its ray.  A warp holds 32 consecutive samples of one ray = 8 Philox
// quads (counter = sample / 4): lanes 0..8 evaluate quads 0..8 once (quad 8: the next warp's first sample), shuffles hand out.
__device__ __forceinline__ void render_jitter_pair(const RenderParams& p, long long s, int lane, bool has_next, float& u0, float& u1) {
  if (p.depth_mode == 1) {
    u0 = u1 = 0.5f;
    return;
  }
  if (p.depth_mode == 0) {
    u0 = p.rand[s];
    u1 = __shfl_down_sync(0xffffffffu, u0, 1);
    if (lane == 31 && has_next) u1 = p.rand[s + 1];
    return;
  }
  const long long qd = ((s - lane) >> 2) + lane;      // (s - lane): the warp's first sample, a multiple of 32
  const uint4 x = tp_philox((uint32_t)qd, (uint32_t)(qd >> 32), (uint32_t)p.seed, (uint32_t)(p.seed >> 32));
  const int src = lane >> 2, e = lane & 3;
  const float c0 = __shfl_sync(0xffffffffu, tp_u01(x.x), src), c1 = __shfl_sync(0xffffffffu, tp_u01(x.y), src),
              c2 = __shfl_sync(0xffffffffu, tp_u01(x.z), src), c3 = __shfl_sync(0xffffffffu, tp_u01(x.w), src);
  u0 = e == 0 ? c0 : e == 1 ? c1 : e == 2 ? c2 : c3;
  const float nq = __shfl_sync(0xffffffffu, tp_u01(x.x), 8);
  u1 = __shfl_down_sync(0xffffffffu, u0, 1);
  if (lane == 31) u1 = nq;
}

template <class P>
__device__ __noinline__ RenderSample render_sample(const P& p, long long tile, int row, int lane) {
  RenderSample o;
  const int N = p.N;                                       // 32, 64 or 128: divides 128
  o.k = row & (N - 1);
  o.ray = render_ray(p, tile, row, o.live);
  long long b, pix;
  float c[3], dir[3];
  render_unproject(p, o.ray, b, pix, c, dir);
  const long long zi = b * (long long)p.H * p.W + pix;
  const float lo = p.z_near[zi], hi = p.z_far[zi];
  float u0, u1;
  render_jitter_pair(p, o.ray * N + o.k, lane, o.k + 1 < N, u0, u1);
  // stratified_depth with N = 2^m: (u + k) / N is an exact scaling, so the multiplication gives the division's bits
  const float inv_n = 1.f / (float)N;
  o.d = __fadd_rn(__fmul_rn(__fmul_rn(__fadd_rn(u0, (float)o.k), inv_n), __fsub_rn(hi, lo)), lo);
  const float dn = __fadd_rn(__fmul_rn(__fmul_rn(__fadd_rn(u1, (float)(o.k + 1)), inv_n), __fsub_rn(hi, lo)), lo);
  const float len = sqrtf(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]);      // composite.cu's |ray|
  o.dist = __fmul_rn(o.k + 1 < N ? __fsub_rn(dn, o.d) : 1e10f, len);
#pragma unroll
  for (int j = 0; j < 3; ++j) o.xyz[j] = __fadd_rn(c[j], __fmul_rn(dir[j], o.d));      // camera.py:317-322
  return o;
}

// The E tile row of the sample: the same fp32 encoding as the per-sample launch's encode_tile (no save slot).
template <bool kSingle, class P>
__device__ __noinline__ void render_encode(const P& p, long long tile, int row, int lane, uint32_t sbase) {
  const RenderSample rs = render_sample(p, tile, row, lane);
  float v[64];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const float x = rs.xyz[j];
    v[j] = x;
#pragma unroll
    for (int k = 0; k < kEncL; ++k) {
      float sn, cs;
      sincosf(__fmul_rn(x, ldexpf(3.14159265358979323846f, k)), &sn, &cs);
      v[3 + j * 2 * kEncL + k] = sn;
      v[3 + j * 2 * kEncL + kEncL + k] = cs;
    }
  }
  v[63] = 0.f;
#pragma unroll
  for (int k8 = 0; k8 < 8; ++k8) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (kSingle) h[e] = pack_bf16(v[k8 * 8 + 2 * e], v[k8 * 8 + 2 * e + 1]);
      else split2(v[k8 * 8 + 2 * e], v[k8 * 8 + 2 * e + 1], h[e], l[e]);
    }
    st_shared_v4(sbase + kOffEhi + k8 * 2048 + row * 16, h[0], h[1], h[2], h[3]);
    if (!kSingle) st_shared_v4(sbase + kOffElo + k8 * 2048 + row * 16, l[0], l[1], l[2], l[3]);
  }
}

// Columns [half * 128, half * 128 + 128) of the rgb-0 bias row of the warp's ray (all 32 rows of a warp share it): imgbias_rgb[view]
// + W_view [u, enc(u)], u = ray / |ray| (layers/nerf_static_transient_light.py:104-117), with tp_tc_ray_bias's operation order --
// one fma chain per column, inputs ascending -- so the row has the table's bits.  Lane j holds input j, lane l computes columns
// 4l .. 4l + 3 of the half; the row goes to the warp's slot `dst`, which the drain of this stage reads back.
template <class P>
__device__ __noinline__ void render_view_row(const P& p, long long tile, int row, int lane, int half, float* dst) {
  bool live;
  const long long ray = render_ray(p, tile, row, live);
  long long b, pix;
  float c[3], dir[3];
  render_unproject(p, ray, b, pix, c, dir);
  const float len = unit_length(dir[0], dir[1], dir[2]);
  const int L = p.L_view, vc = 3 + 6 * L;
  float e = 0.f;
  if (lane < vc) {
    const int jj = lane - 3, cc = lane < 3 ? lane : jj / (2 * L);
    const float uc = __fdiv_rn(cc == 0 ? dir[0] : cc == 1 ? dir[1] : dir[2], len);
    e = uc;
    if (lane >= 3) {
      const int rem = jj - cc * 2 * L, k = rem < L ? rem : rem - L;
      const float arg = __fmul_rn(uc, ldexpf(3.14159265358979323846f, k));
      e = rem < L ? sinf(arg) : cosf(arg);
    }
  }
  const int col = half * 128 + lane * 4;
  float4 acc = __ldg(reinterpret_cast<const float4*>(p.imgbias_rgb + b * 256 + col));
  // inputs nine at a time: the nine weight loads of a batch are independent (one L2 round trip per batch, not per input)
#pragma unroll 1
  for (int j0 = 0; j0 < vc; j0 += 9) {
    float4 w[9];
#pragma unroll
    for (int i = 0; i < 9; ++i)
      if (j0 + i < vc) w[i] = __ldg(reinterpret_cast<const float4*>(p.wview + (j0 + i) * 256 + col));
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      const float ej = __shfl_sync(0xffffffffu, e, (j0 + i) & 31);
      if (j0 + i < vc) {
        acc.x = fmaf(w[i].x, ej, acc.x);
        acc.y = fmaf(w[i].y, ej, acc.y);
        acc.z = fmaf(w[i].z, ej, acc.z);
        acc.w = fmaf(w[i].w, ej, acc.w);
      }
    }
  }
  *reinterpret_cast<float4*>(dst + lane * 4) = acc;
}

__device__ __forceinline__ float warp_scan(float v, int lane) {      // inclusive
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float n = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += n;
  }
  return v;
}

// Compositing of the tile's rays by the four column-half-0 warps (rows = samples; N / 32 warps per ray), arithmetic of
// tp_composite_stl_forward (layers/nerf_static_transient_light.py:168-212, SURVEY appendix C): three exclusive cumulative sums
// (warp scan + the totals of the ray's earlier warps, exchanged through `sc`), 14 per-ray sums (warp reduction + the same
// exchange).  The plain model (layers/nerf.py:117-136) is the same arithmetic with a zero transient head: sig_t = 0 makes the
// joint and static chains equal, rgb = sum c w, depth = sum d w, opacity = sum w with w = T (1 - exp(-sigma dist)) -- the weights
// of tp_composite_plain_forward.
__device__ __noinline__ void render_composite(const RenderParams& p, float* sc, int q, int lane, long long ray, int k, float d,
                                              float dist, bool live, float sig_s, float sig_t, float cs0, float cs1, float cs2,
                                              float ct0, float ct1, float ct2, float u) {
  const float cs[3] = {cs0, cs1, cs2}, ct[3] = {ct0, ct1, ct2};
  float* tot = sc;             // [4 warps][3]
  float* red = sc + 12;        // [4 warps][14]
  const float sd_s = __fmul_rn(sig_s, dist), sd_t = __fmul_rn(sig_t, dist), sd = __fadd_rn(sd_s, sd_t);
  const float in_j = warp_scan(sd, lane), in_s = warp_scan(sd_s, lane), in_t = warp_scan(sd_t, lane);
  if (lane == 31) {
    tot[q * 3] = in_j;
    tot[q * 3 + 1] = in_s;
    tot[q * 3 + 2] = in_t;
  }
  const float pj = __shfl_up_sync(0xffffffffu, in_j, 1), ps_ = __shfl_up_sync(0xffffffffu, in_s, 1),
              pt_ = __shfl_up_sync(0xffffffffu, in_t, 1);
  named_bar_sync(1, 128);
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
  float v16[16];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    v16[c] = cs[c] * w_ps + ct[c] * w_pt;
    v16[3 + c] = w_qs * cs[c];
    v16[6 + c] = w_qt * ct[c];
  }
  v16[9] = d * w_qs;
  v16[10] = w_p;
  v16[11] = w_qs;
  v16[12] = w_qt;
  v16[13] = u * w_pt;
  v16[14] = v16[15] = 0.f;
  // warp totals of the 16 values by recursive halving (8 + 4 + 2 + 1 + 1 shuffles): a lane keeps one half and adds the partner's
  float v8[8], v4[4], v2[2];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const bool up = (lane & 16) != 0;
    v8[i] = (up ? v16[i + 8] : v16[i]) + __shfl_xor_sync(0xffffffffu, up ? v16[i] : v16[i + 8], 16);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool up = (lane & 8) != 0;
    v4[i] = (up ? v8[i + 4] : v8[i]) + __shfl_xor_sync(0xffffffffu, up ? v8[i] : v8[i + 4], 8);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const bool up = (lane & 4) != 0;
    v2[i] = (up ? v4[i + 2] : v4[i]) + __shfl_xor_sync(0xffffffffu, up ? v4[i] : v4[i + 2], 4);
  }
  const bool up2 = (lane & 2) != 0;
  float v1 = (up2 ? v2[1] : v2[0]) + __shfl_xor_sync(0xffffffffu, up2 ? v2[0] : v2[1], 2);
  v1 += __shfl_xor_sync(0xffffffffu, v1, 1);
  const int vidx = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
  if ((lane & 1) == 0 && vidx < 14) red[q * 14 + vidx] = v1;
  if (live) {
    const long long s = ray * p.N + k;
    if (p.o_as) __stcs(p.o_as + s, as);
    if (p.o_at) __stcs(p.o_at + s, at);
    if (p.o_density) {
      if (p.chains == 1) __stcs(p.o_density + s, sig_s);
      else __stcs(reinterpret_cast<float2*>(p.o_density) + s, make_float2(sig_s, sig_t));
    }
  }
  named_bar_sync(1, 128);
  if (q == q0 && lane < 14 && live) {
    float v = 0.f;
    for (int w = q0; w < q0 + wpr; ++w) v += red[w * 14 + lane];
    float* dst = lane < 3 ? (p.o_rgb ? p.o_rgb + ray * 3 + lane : nullptr)
               : lane < 6 ? (p.o_rgb_s ? p.o_rgb_s + ray * 3 + lane - 3 : nullptr)
               : lane < 9 ? (p.o_rgb_t ? p.o_rgb_t + ray * 3 + lane - 6 : nullptr)
               : lane == 9 ? (p.o_depth ? p.o_depth + ray : nullptr)
               : lane == 10 ? (p.o_op ? p.o_op + ray : nullptr)
               : lane == 11 ? (p.o_op_s ? p.o_op_s + ray : nullptr)
               : lane == 12 ? (p.o_op_t ? p.o_op_t + ray : nullptr)
                            : (p.o_unc ? p.o_unc + ray : nullptr);
    if (lane == 13) v += p.min_uncert;
    if (dst) *dst = v;
  }
}

// kSingle = false: the fp32-parity mode (fp16 hi + lo, three passes).  kSingle = true: ONE pass with bf16 operands -- the general-
// architecture bf16 forward (any stage list; <= 1e-2 like mlp_tc.cu, which stays the fast path for the yaml's architecture), whose
// drain can also keep every hidden activation as a bf16 tile image for the tensor-core backward (training of layers/nerf.py).
// kSplitSave (with kSingle = false): the parity-mode arithmetic unchanged, and the drain also keeps every save-slot activation and
// the encoding tile as bf16 hi + lo tile images (slots 2k, 2k + 1) plus the ReLU bitmasks: the operands of the split backward.
// P = RenderParams: the render launch (samples made in-kernel, per-ray outputs; no save); P = ListRenderParams: the same over an
// object-pixel list, this rank's share of its tiles.
template <bool kSingle, bool kSplitSave, class P = Params>
__device__ __forceinline__ void nerf_forward_split_body(const P& p) {
  static_assert(!(kSingle && kSplitSave), "the split save belongs to the three-pass arithmetic");
  constexpr bool kRender = std::is_base_of<RenderParams, P>::value;
  static_assert(!(kRender && kSplitSave), "the render launch keeps no activations");
  constexpr bool kSave = (kSingle || kSplitSave) && !kRender;      // the launch can write tile images
  constexpr int kImgPerSlot = kSplitSave ? 2 : 1;     // tile images per save slot (hi, lo)
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const uint32_t bar0 = sbase + kOffBar;
  auto bar_full = [&](int s) { return bar0 + 8 * s; };
  auto bar_empty = [&](int s) { return bar0 + 8 * (kRing + s); };
  auto bar_acc = [&](int i) { return bar0 + 8 * (2 * kRing + i); };
  auto bar_ready = [&](int g) { return bar0 + 8 * (2 * kRing + 2 + g); };          // 8: A columns [32g, 32g+32) written
  auto bar_reload = [&](int g) { return bar0 + 8 * (2 * kRing + 10 + g); };        // 8: parked feature columns back in A
  const uint32_t bar_enc = bar0 + 8 * (2 * kRing + 18), bar_out = bar_enc + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffBar + 8 * (2 * kRing + 20));

  if (threadIdx.x == 0) {
    for (int s = 0; s < kRing; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_empty(s), 1);
    }
    mbar_init(bar_acc(0), 1);
    mbar_init(bar_acc(1), 1);
    for (int g = 0; g < 8; ++g) {
      mbar_init(bar_ready(g), 4);        // the four lane-quarter warps of the column half
      mbar_init(bar_reload(g), 1);
    }
    mbar_init(bar_enc, 4);
    mbar_init(bar_out, 4);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const long long n_tiles = launch_tiles(p);
  const int n_stages = p.n_stages;

  if (warp == kProducerWarp) {
    // ================================================================ weight producer
    uint32_t slot = 0, phase = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      long long c = 0;
      for (int L = 0; L < n_stages; ++L) {
        const Stage sg = p.st[L];
        const bool small = sg.kind != KIND_HIDDEN;
        const int n = small ? 1 : sg.e_steps + sg.a_steps;
        const uint32_t bytes = (small || kSingle) ? kHalfSlot : kSlotBytes;      // single pass: only the hi half of a slot exists
        for (int j = 0; j < n; ++j, ++c) {
          mbar_wait(bar_empty(slot), phase ^ 1);
          if (elect_one_sync()) {
            mbar_expect_tx(bar_full(slot), bytes);
            bulk_g2s_hint(sbase + kOffRing + slot * kSlotBytes, p.image + (size_t)c * kSlotBytes, bytes, bar_full(slot),
                          l2_policy_evict_last());
          }
          __syncwarp();
          if (++slot == kRing) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ================================================================ MMA issuer
    uint32_t slot = 0, phase = 0, ready_ph = 0, reload_ph = 0, enc_ph = 0, out_ph = 0;
    const uint32_t idesc256 = kSingle ? umma_idesc(128, 256) : umma_idesc_f16(128, 256);
    const uint32_t idesc16 = kSingle ? umma_idesc(128, 16) : umma_idesc_f16(128, 16);
    constexpr uint32_t kHi = (128u >> 4) | (1u << 14);      // SBO = 128 B, descriptor version 1
    bool first_tile = true;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      mbar_wait(bar_enc, enc_ph);            // the tile's encoding is in E
      enc_ph ^= 1;
      if (!first_tile) {                     // the previous tile's last accumulator has been read
        mbar_wait(bar_out, out_ph);
        out_ph ^= 1;
      }
      first_tile = false;
      for (int L = 0; L < n_stages; ++L) {
        const Stage sg = p.st[L];
        const uint32_t d_tmem = tmem_base + (uint32_t)(L & 1) * 256;
        const bool wait_ready = (sg.flags & F_WAIT_READY) != 0, reload = (sg.flags & F_RELOAD) != 0;
        if (sg.kind == KIND_HIDDEN) {
          const int n = sg.e_steps + sg.a_steps;
          for (int step = 0; step < n; ++step) {
            const bool from_e = step < sg.e_steps;
            const int ks = from_e ? step : step - sg.e_steps;
            if (!from_e && (ks & 1) == 0) {
              if (reload) mbar_wait(bar_reload(ks >> 1), reload_ph);
              else if (wait_ready) mbar_wait(bar_ready(ks >> 1), ready_ph);
            }
            mbar_wait(bar_full(slot), phase);
            tc_fence_after();
            if (elect_one_sync()) {
              const uint32_t wsm = sbase + kOffRing + slot * kSlotBytes;
              const uint32_t bh = (wsm >> 4) | ((4096u >> 4) << 16), bl = ((wsm + kHalfSlot) >> 4) | ((4096u >> 4) << 16);
              const uint32_t a0 = (from_e ? kOffEhi : kOffAhi) + (uint32_t)ks * 4096u;
              const uint32_t a1 = (from_e ? kOffElo : kOffAlo) + (uint32_t)ks * 4096u;
              const uint32_t ah = ((sbase + a0) >> 4) | ((2048u >> 4) << 16), al = ((sbase + a1) >> 4) | ((2048u >> 4) << 16);
              if (kSingle) umma_bf16_lohi(d_tmem, ah, kHi, bh, kHi, idesc256, step > 0 ? 1u : 0u);
              else umma3(d_tmem, ah, al, kHi, bh, bl, kHi, idesc256, step > 0 ? 1u : 0u);
              umma_commit(bar_empty(slot));
              if (step == n - 1) umma_commit(bar_acc(L & 1));
            }
            __syncwarp();
            if (++slot == kRing) { slot = 0; phase ^= 1; }
          }
        } else {
          // N = 16 output stage: one 8 KB slot [32 k8][16 rows][8] spans K = 256; pass 0 reads A_hi, pass 1 A_lo
          mbar_wait(bar_full(slot), phase);
          const uint32_t wsm = sbase + kOffRing + slot * kSlotBytes;
          for (int ks = 0; ks < 16; ++ks) {
            if ((ks & 1) == 0) {
              if (reload) mbar_wait(bar_reload(ks >> 1), reload_ph);
              else if (wait_ready) mbar_wait(bar_ready(ks >> 1), ready_ph);
            }
            tc_fence_after();
            if (elect_one_sync()) {
              const uint32_t ah = ((sbase + kOffAhi + (uint32_t)ks * 4096u) >> 4) | ((2048u >> 4) << 16);
              const uint32_t b = ((wsm + (uint32_t)ks * 512u) >> 4) | ((256u >> 4) << 16);
              umma_bf16_lohi(d_tmem, ah, kHi, b, kHi, idesc16, ks > 0 ? 1u : 0u);
            }
            __syncwarp();
          }
          if (elect_one_sync()) {
            if (!kSingle) {
#pragma unroll
              for (int ks = 0; ks < 16; ++ks) {
                const uint32_t al = ((sbase + kOffAlo + (uint32_t)ks * 4096u) >> 4) | ((2048u >> 4) << 16);
                const uint32_t b = ((wsm + (uint32_t)ks * 512u) >> 4) | ((256u >> 4) << 16);
                umma_bf16_lohi(d_tmem, al, kHi, b, kHi, idesc16, 1u);
              }
            }
            umma_commit(bar_empty(slot));
            umma_commit(bar_acc(L & 1));
          }
          __syncwarp();
          if (++slot == kRing) { slot = 0; phase ^= 1; }
        }
        if (reload) reload_ph ^= 1;
        else if (wait_ready) ready_ph ^= 1;
      }
    }
  } else {
    // ================================================================ drain / encode warps
    // warp -> (TMEM lane quarter q, column half): each thread converts 128 accumulator columns of its row
    const int q = warp & 3, half = warp >> 2, row = q * 32 + lane;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16);
    uint8_t* park = p.scratch + (size_t)blockIdx.x * 2 * kABytes;
    uint32_t acc_ph = 0;      // bit i: phase of bar_acc(i)
    float act_max = 0.f;      // split mode: largest hidden activation this thread converted (fp16 hi saturates at 65 504)

    // fp32 encoding of one sample (layers/nerf_static_transient_light.py:217-234: the reference multiplies by fl(2^k pi) and
    // takes sin / cos of the ROUNDED product -- its own encoding differs from the exact one by up to 6e-5 at k = 9, so the
    // parity mode must round where it rounds), split into E_hi / E_lo.  Done by the column-half-1 warps (row = sample).
    auto encode_tile = [&](long long tile) {
      if constexpr (kRender) {
        render_encode<kSingle>(p, tile, row, lane, sbase);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_enc);
        return;
      }
      const long long s_raw = tile * 128 + row, s = s_raw < p.S ? s_raw : p.S - 1, r = s / p.N;
      const float d = p.depth[s];
      float v[64];
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const float x = __fadd_rn(p.center[r * 3 + j], __fmul_rn(p.ray[r * 3 + j], d));      // camera.py:317-322
        v[j] = x;
#pragma unroll
        for (int k = 0; k < kEncL; ++k) {
          float sn, cs;
          sincosf(__fmul_rn(x, ldexpf(3.14159265358979323846f, k)), &sn, &cs);
          v[3 + j * 2 * kEncL + k] = sn;
          v[3 + j * 2 * kEncL + kEncL + k] = cs;
        }
      }
      uint8_t* const g_enc = (kSave && p.save && p.enc_slot >= 0)
                                 ? p.save + ((size_t)tile * kImgPerSlot * p.n_save + kImgPerSlot * p.enc_slot) * kABytes + row * 16
                                 : nullptr;
      v[63] = g_enc ? 1.f : 0.f;      // (no layer has a weight column 63: the packed images hold zeros there)
#pragma unroll
      for (int k8 = 0; k8 < 8; ++k8) {
        uint32_t h[4], l[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (kSingle) h[e] = pack_bf16(v[k8 * 8 + 2 * e], v[k8 * 8 + 2 * e + 1]);
          else split2(v[k8 * 8 + 2 * e], v[k8 * 8 + 2 * e + 1], h[e], l[e]);
        }
        st_shared_v4(sbase + kOffEhi + k8 * 2048 + row * 16, h[0], h[1], h[2], h[3]);
        if (!kSingle) st_shared_v4(sbase + kOffElo + k8 * 2048 + row * 16, l[0], l[1], l[2], l[3]);
        if (kSplitSave && g_enc) {
#pragma unroll
          for (int e = 0; e < 4; ++e) split2_bf16(v[k8 * 8 + 2 * e], v[k8 * 8 + 2 * e + 1], h[e], l[e]);
          st_global_cs_v4(g_enc + k8 * 2048, h[0], h[1], h[2], h[3]);
          st_global_cs_v4(g_enc + kABytes + k8 * 2048, l[0], l[1], l[2], l[3]);
        } else if (g_enc) {
          st_global_cs_v4(g_enc + k8 * 2048, h[0], h[1], h[2], h[3]);
        }
      }
      if (g_enc) {
#pragma unroll 4
        for (int k8 = 8; k8 < 32; ++k8) st_global_cs_v4(g_enc + k8 * 2048, 0u, 0u, 0u, 0u);
        if (kSplitSave) {
#pragma unroll 4
          for (int k8 = 8; k8 < 32; ++k8) st_global_cs_v4(g_enc + kABytes + k8 * 2048, 0u, 0u, 0u, 0u);
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_enc);
    };
    if (half == 1 && (long long)blockIdx.x < n_tiles) encode_tile(blockIdx.x);
    float* vrow = nullptr;      // render launch: this warp's slot for its half of the rgb-0 bias row
    if constexpr (kRender) vrow = reinterpret_cast<float*>(p.scratch + p.vrow_off) + ((size_t)blockIdx.x * 8 + warp) * kViewRowFloats;

    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const long long s_raw = tile * 128 + row;
      const bool live = s_raw < p.S;
      const long long s = live ? s_raw : p.S - 1;
      float sigma_s = 0.f, rgb_s[3] = {0.f, 0.f, 0.f}, rgb_t[3] = {0.f, 0.f, 0.f}, sigma_t = 0.f, unc = 0.f;
      for (int L = 0; L < n_stages; ++L) {
        const Stage sg = p.st[L];
        if constexpr (kRender) {
          if (sg.bias_kind == BIAS_RAY) {      // while the stage's MMAs run: the warp's half of its ray's bias row
            render_view_row(p, tile, row, lane, half, vrow);
            __syncwarp();
          }
        }
        mbar_wait(bar_acc(L & 1), (acc_ph >> (L & 1)) & 1u);
        acc_ph ^= 1u << (L & 1);
        tc_fence_after();
        if (L + 1 < n_stages && (p.st[L + 1].flags & F_RELOAD) && threadIdx.x == 0) {
          // every MMA that read A has retired: bring the parked feature back, one 32-column group (hi + lo) per barrier
          fence_proxy_async_all();
#pragma unroll 1
          for (int g = 0; g < 8; ++g) {
            mbar_expect_tx(bar_reload(g), kSingle ? kHalfSlot : 2 * kHalfSlot);
            bulk_g2s(sbase + kOffAhi + g * kHalfSlot, park + g * kHalfSlot, kHalfSlot, bar_reload(g));
            if (!kSingle) bulk_g2s(sbase + kOffAlo + g * kHalfSlot, park + kABytes + g * kHalfSlot, kHalfSlot, bar_reload(g));
          }
        }
        if (sg.kind == KIND_HIDDEN) {
          const float* brow = kRender && sg.bias_kind == BIAS_RAY ? vrow
                            : (sg.bias_kind == BIAS_STATIC ? p.bias + sg.bias_off
                               : sg.bias_kind == BIAS_RAY  ? p.raybias + (s / p.N) * 256
                                                           : p.imgbias + image_of(p, tile, row, s) * 256) + half * 128;
          const uint32_t tmem_d = tmem_row + (uint32_t)(L & 1) * 256 + half * 128;
          const bool do_park = (sg.flags & F_PARK) != 0;
          uint8_t* const g_save = (kSave && p.save && sg.save_slot >= 0)
                                      ? p.save + ((size_t)tile * kImgPerSlot * p.n_save + kImgPerSlot * sg.save_slot) * kABytes
                                      : nullptr;
          uint32_t* const g_bits = g_save ? p.save_bits + ((size_t)tile * p.n_save + sg.save_slot) * 1024 + half * 4 * 128 + row : nullptr;
          // one 32-column slab: + bias, ReLU, hi / lo split, 4 core-matrix rows of A_hi and A_lo (and of the parked copy)
          // the slab's 32 bias values are fetched one slab ahead (beside the TMEM load): loads issued inside the conversion loop
          // wait out their full latency behind the stores of the previous group (16 exposed load-use stalls per stage, ncu source page)
          auto load_bias = [&](float4 (&bq)[8], int j) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4* a = reinterpret_cast<const float4*>(brow + j * 32 + i * 4);
              bq[i] = kRender ? __ldcg(a) : __ldg(a);      // (the render launch's bias row was written by this kernel)
            }
          };
          auto slab = [&](const uint32_t (&v)[32], const float4 (&bq)[8], int j) {
            uint32_t positive = 0u;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 b0 = bq[2 * i], b1 = bq[2 * i + 1];
              const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
              uint32_t h[4], l[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float x0 = __uint_as_float(v[i * 8 + 2 * e]) + bb[2 * e], x1 = __uint_as_float(v[i * 8 + 2 * e + 1]) + bb[2 * e + 1];
                if (kSingle) {
                  h[e] = pack_relu_bf16(x0, x1);
                  if (g_save) {      // sign bits, first column shifted in first (one funnel shift per element; reversed below)
                    positive = __funnelshift_l(__float_as_uint(x0), positive, 1);
                    positive = __funnelshift_l(__float_as_uint(x1), positive, 1);
                  }
                } else {
                  split2(fmaxf(x0, 0.f), fmaxf(x1, 0.f), h[e], l[e]);
                  act_max = fmaxf(act_max, fmaxf(x0, x1));
                }
              }
              const uint32_t off = (uint32_t)(half * 16 + j * 4 + i) * 2048 + row * 16;
              st_shared_v4(sbase + kOffAhi + off, h[0], h[1], h[2], h[3]);
              if (!kSingle) st_shared_v4(sbase + kOffAlo + off, l[0], l[1], l[2], l[3]);
              if (do_park) {
                st_global_v4(park + off, h[0], h[1], h[2], h[3]);
                if (!kSingle) st_global_v4(park + kABytes + off, l[0], l[1], l[2], l[3]);
              }
              if (kSplitSave && g_save) {      // (recomputed here, after the fp16 words are stored: fewer live registers)
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float x0 = __uint_as_float(v[i * 8 + 2 * e]) + bb[2 * e], x1 = __uint_as_float(v[i * 8 + 2 * e + 1]) + bb[2 * e + 1];
                  split2_bf16(fmaxf(x0, 0.f), fmaxf(x1, 0.f), h[e], l[e]);
                  positive = __funnelshift_l(__float_as_uint(x0), positive, 1);
                  positive = __funnelshift_l(__float_as_uint(x1), positive, 1);
                }
                st_global_cs_v4(g_save + off, h[0], h[1], h[2], h[3]);
                st_global_cs_v4(g_save + kABytes + off, l[0], l[1], l[2], l[3]);
              } else if (g_save) {
                st_global_cs_v4(g_save + off, h[0], h[1], h[2], h[3]);
              }
            }
            if (g_bits) g_bits[j * 128] = __brev(~positive);      // bit c = column c of the slab is positive (sign bit clear)
            if (do_park) __threadfence();      // the parked copy is read back through the async proxy (bulk load) four stages later
            fence_proxy_async_smem();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_ready(half * 4 + j));
          };
          uint32_t va[32], vb[32];
          float4 ba[8], bb2[8];
          TP_TMEM_LD32(tmem_d, va);
          load_bias(ba, 0);
          TP_TMEM_WAIT32(va);
          TP_TMEM_LD32(tmem_d + 32, vb);
          load_bias(bb2, 1);
          slab(va, ba, 0);
          TP_TMEM_WAIT32(vb);
          TP_TMEM_LD32(tmem_d + 64, va);
          load_bias(ba, 2);
          slab(vb, bb2, 1);
          TP_TMEM_WAIT32(va);
          TP_TMEM_LD32(tmem_d + 96, vb);
          load_bias(bb2, 3);
          slab(va, ba, 2);
          TP_TMEM_WAIT32(vb);
          slab(vb, bb2, 3);
          if ((sg.flags & F_E_LAST) && half == 1 && tile + gridDim.x < n_tiles) encode_tile(tile + gridDim.x);
        } else if (half == 0) {
          uint32_t v[16];
          TP_TMEM_LD16(tmem_row + (uint32_t)(L & 1) * 256, v);
          TP_TMEM_WAIT16(v);
          if (L == n_stages - 1) {           // the next tile's first stage may overwrite this accumulator
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_out);
          }
          const float* sb = p.bias + sg.bias_off;
          auto out = [&](int c) { return __uint_as_float(v[c]) + __uint_as_float(v[c + 8]) + sb[c]; };
          if (sg.kind == KIND_DENSITY) {
            sigma_s = tp_softplus(out(0));
          } else if (sg.kind == KIND_RGB_OUT) {
#pragma unroll
            for (int c = 0; c < 3; ++c) rgb_s[c] = tp_sigmoid(out(c));
          } else {
#pragma unroll
            for (int c = 0; c < 3; ++c) rgb_t[c] = tp_sigmoid(out(c));
            sigma_t = tp_softplus(out(3));
            unc = tp_softplus(out(4));
          }
        }
      }
      if (!kSingle && !(act_max <= 6.0e4f)) atomicOr(p.status, 1u);      // (also catches NaN)
      if constexpr (kRender) {
        if (half == 0) {
          const RenderSample rs = render_sample(p, tile, row, lane);
          render_composite(p, reinterpret_cast<float*>(smem + kOffComp), q, lane, rs.ray, rs.k, rs.d, rs.dist, rs.live, sigma_s,
                           sigma_t, rgb_s[0], rgb_s[1], rgb_s[2], rgb_t[0], rgb_t[1], rgb_t[2], unc);
        }
      } else if (half == 0 && live) {
#pragma unroll
        for (int c = 0; c < 3; ++c) *reinterpret_cast<float2*>(p.rgb + s * 6 + c * 2) = make_float2(rgb_s[c], rgb_t[c]);
        *reinterpret_cast<float2*>(p.density + s * 2) = make_float2(sigma_s, sigma_t);
        p.uncert[s] = unc;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

template <bool kSingle>
__global__ void __launch_bounds__(kThreads, 1) nerf_forward_split_kernel(const Params p) {
  nerf_forward_split_body<kSingle, false>(p);
}
// the parity-mode forward of a training step: tile images and ReLU bitmasks in the split backward's format
__global__ void __launch_bounds__(kThreads, 1) nerf_forward_split_save_kernel(const Params p) {
  nerf_forward_split_body<false, true>(p);
}

// the render launch in either arithmetic
template <bool kSingle>
__global__ void __launch_bounds__(kThreads, 1) nerf_render_split_kernel(const __grid_constant__ RenderParams p) {
  nerf_forward_split_body<kSingle, false, RenderParams>(p);
}
template <bool kSingle>
__global__ void __launch_bounds__(kThreads, 1) nerf_render_list_split_kernel(const __grid_constant__ ListRenderParams p) {
  nerf_forward_split_body<kSingle, false, ListRenderParams>(p);
}

// slot_desc row: [W ptr, ld, row0, rows_valid, col0, cols_valid, kind (256 | 16), unused]
//   kind 256: slot = [hi | lo], each [2 k8][256 rows][8]: element (n, kl) = W[row0 + n][col0 + kl], kl < 16
//   kind 16:  first 8 KB = [32 k8][16 rows][8]: rows 0..7 hi, rows 8..15 lo of W[row0 + (n & 7)][col0 + kl], kl < 256
// bf16 != 0: the single-pass image -- bf16(W) in the hi half (the lo half stays zero and is never streamed); output layers keep
// their hi / lo rows, as bf16
__global__ void pack_split_kernel(const long long* __restrict__ desc, uint16_t* __restrict__ out, int bf16) {
  const long long* d = desc + (long long)blockIdx.x * 8;
  const float* W = reinterpret_cast<const float*>(d[0]);
  const long long ld = d[1], row0 = d[2], rows_valid = d[3], col0 = d[4], cols_valid = d[5], kind = d[6];
  uint16_t* o = out + (long long)blockIdx.x * (kSlotBytes / 2);
  for (int e = threadIdx.x; e < (int)(kSlotBytes / 2); e += blockDim.x) {
    int n, kl;
    bool lo_part, in_layout = true;
    if (kind == 256) {
      lo_part = e >= 4096;
      const int f = e & 4095;
      kl = (f >> 11) * 8 + (f & 7);
      n = (f >> 3) & 255;
    } else {
      in_layout = e < 4096;
      kl = (e >> 7) * 8 + (e & 7);
      n = (e >> 3) & 15;
      lo_part = n >= 8;
      n &= 7;
    }
    float v = 0.f;
    if (in_layout && W && n < rows_valid && kl < cols_valid) v = W[(row0 + n) * ld + col0 + kl];
    if (bf16) {
      if (lo_part) v = kind == 256 ? 0.f : v - __bfloat162float(__float2bfloat16_rn(v));
      o[e] = __bfloat16_as_ushort(__float2bfloat16_rn(v));
    } else {
      if (lo_part) v -= __half2float(__float2half_rn(v));
      o[e] = __half_as_ushort(__float2half_rn(v));
    }
  }
}

}  // namespace tcs

TP_API int64_t tp_tc32_slot_bytes(void) { return tcs::kSlotBytes; }
/* bytes of the save buffer of a single-pass launch: [tiles][n_save][64 KB] tile images, then [tiles][n_save][4 KB] ReLU bitmasks */
TP_API int64_t tp_tc32_save_bytes(int64_t S, int n_save) { return ((S + 127) / 128) * (int64_t)n_save * (tc::kABytes + 4096); }
TP_API int64_t tp_tc32_scratch_bytes(void) { return (int64_t)tp_num_sms() * 2 * tc::kABytes + 16; }
TP_API int64_t tp_tc32_status_offset(void) { return (int64_t)tp_num_sms() * 2 * tc::kABytes; }
TP_API int tp_tc32_max_stages(void) { return tcs::kMaxStages; }

TP_API int tp_tc32_pack_weights(const int64_t* slot_desc, int n_slots, int precision, void* image, void* stream) {
  if (!slot_desc || !image) return TP_ERR_BAD_ARG;
  if (n_slots < 1) return TP_ERR_BAD_SHAPE;
  if (precision != 0 && precision != 1) return TP_ERR_BAD_ARG;
  tcs::pack_split_kernel<<<n_slots, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const long long*>(slot_desc),
                                                                   reinterpret_cast<uint16_t*>(image), precision);
  return tp_launch_status();
}

/* bytes of the save buffer of a split-save launch: [tiles][2 n_save][64 KB] hi / lo tile images, then [tiles][n_save][4 KB] bitmasks */
TP_API int64_t tp_tc32_split_save_bytes(int64_t S, int n_save) {
  return ((S + 127) / 128) * (int64_t)n_save * (2 * tc::kABytes + 4096);
}

// The stage list into p.st: it is the caller's architecture, and a malformed list would dead-lock the barrier protocol.
// has_raybias / has_imgbias: the launch has the per-ray / per-image bias rows that BIAS_RAY / BIAS_IMAGE stages read.
static int tc32_parse_stages(tcs::Params& p, const int32_t* stages, int n_stages, int n_slots, bool has_raybias, bool has_imgbias,
                             const void* save, int n_save, int enc_slot) {
  int slots = 0, pending_ready = 0, n_e_last = 0;
  bool parked = false;
  for (int L = 0; L < n_stages; ++L) {
    tcs::Stage& sg = p.st[L];
    const int32_t* r = stages + L * 7;
    sg.a_steps = r[0]; sg.e_steps = r[1]; sg.kind = r[2]; sg.bias_kind = r[3]; sg.bias_off = r[4]; sg.flags = r[5]; sg.save_slot = r[6];
    if (sg.save_slot < -1 || (save && sg.save_slot >= n_save) || (sg.save_slot >= 0 && sg.kind != tcs::KIND_HIDDEN)) return TP_ERR_BAD_ARG;
    if (sg.save_slot >= 0 && sg.save_slot == enc_slot) return TP_ERR_BAD_ARG;
    if (sg.kind < 0 || sg.kind > 3 || sg.bias_kind < 0 || sg.bias_kind > 2 || sg.bias_off < 0 || (sg.bias_off & 3)) return TP_ERR_BAD_ARG;
    if (sg.e_steps < 0 || sg.e_steps > 4 || (sg.a_steps != 0 && sg.a_steps != 16)) return TP_ERR_BAD_SHAPE;
    const bool hidden = sg.kind == tcs::KIND_HIDDEN, wait = sg.flags & tcs::F_WAIT_READY, reload = sg.flags & tcs::F_RELOAD;
    if (!hidden && (sg.a_steps != 16 || sg.e_steps != 0 || sg.bias_kind != tcs::BIAS_STATIC)) return TP_ERR_BAD_SHAPE;
    if (hidden && sg.a_steps + sg.e_steps == 0) return TP_ERR_BAD_SHAPE;
    if ((wait || reload) && sg.a_steps != 16) return TP_ERR_BAD_ARG;
    if (wait && reload) return TP_ERR_BAD_ARG;
    if (wait && pending_ready != 1) return TP_ERR_BAD_ARG;              // exactly one drain's arrivals are outstanding
    if (wait) pending_ready = 0;
    if (reload && (!parked || L == 0 || p.st[L - 1].kind == tcs::KIND_HIDDEN || pending_ready)) return TP_ERR_BAD_ARG;
    if (sg.a_steps && !wait && !reload && (L == 0 || p.st[L - 1].kind == tcs::KIND_HIDDEN)) return TP_ERR_BAD_ARG;   // A would be stale
    if (sg.bias_kind == tcs::BIAS_RAY && !has_raybias) return TP_ERR_BAD_ARG;
    if (sg.bias_kind == tcs::BIAS_IMAGE && !has_imgbias) return TP_ERR_BAD_ARG;
    if (hidden) {
      if (pending_ready) return TP_ERR_BAD_ARG;                          // the previous drain's arrivals were never consumed
      pending_ready = 1;
      if (sg.flags & tcs::F_PARK) parked = true;
    }
    if (sg.flags & tcs::F_E_LAST) ++n_e_last;
    slots += hidden ? sg.a_steps + sg.e_steps : 1;
  }
  for (int L = 0, seen = 0; L < n_stages; ++L) {      // E_LAST marks the last stage that reads E, and a hidden one
    if (p.st[L].flags & tcs::F_E_LAST) seen = 1;
    else if (seen && p.st[L].e_steps) return TP_ERR_BAD_ARG;
    if ((p.st[L].flags & tcs::F_E_LAST) && p.st[L].kind != tcs::KIND_HIDDEN) return TP_ERR_BAD_ARG;
  }
  if (n_e_last != 1 || pending_ready || p.st[0].e_steps == 0 || p.st[n_stages - 1].kind == tcs::KIND_HIDDEN) return TP_ERR_BAD_ARG;
  if (slots != n_slots) return TP_ERR_BAD_SHAPE;
  p.n_stages = n_stages;
  return TP_OK;
}

// shared by tp_tc32_forward and tp_tc32_forward_split_save: the argument and stage-list checks, then the launch
static int tc32_forward_launch(const float* center, const float* ray, const float* depth, int64_t S, int N, int64_t per_image,
                               const void* image, int n_slots, const int32_t* stages, int n_stages, const float* bias,
                               const float* raybias, const float* imgbias, float* rgb, float* density, float* uncert,
                               void* scratch, int64_t scratch_bytes, int precision, void* save, int n_save, int enc_slot,
                               bool split_save, void* stream) {
  if (enc_slot < -1 || (enc_slot >= 0 && (!save || enc_slot >= n_save))) return TP_ERR_BAD_ARG;
  if (((uintptr_t)image & 15) || ((uintptr_t)scratch & 15) || ((uintptr_t)bias & 15) || ((uintptr_t)raybias & 15) ||
      ((uintptr_t)imgbias & 15) || ((uintptr_t)rgb & 7) || ((uintptr_t)density & 7))
    return TP_ERR_ALIGN;
  if (!tp_device_is_sm100()) return TP_ERR_ARCH;
  tcs::Params p = {};
  const int err = tc32_parse_stages(p, stages, n_stages, n_slots, raybias != nullptr, imgbias != nullptr, save, n_save, enc_slot);
  if (err != TP_OK) return err;
  if (S == 0) return TP_OK;
  const long long n_tiles = (S + 127) / 128;
  int grid = tp_num_sms();
  if (n_tiles < grid) grid = (int)n_tiles;
  if (scratch_bytes < tp_tc32_scratch_bytes()) return TP_ERR_WORKSPACE;
  p.center = center; p.ray = ray; p.depth = depth; p.S = S; p.N = N; p.per_image = per_image;
  p.image = reinterpret_cast<const uint8_t*>(image); p.bias = bias; p.raybias = raybias; p.imgbias = imgbias;
  p.rgb = rgb; p.density = density; p.uncert = uncert; p.scratch = reinterpret_cast<uint8_t*>(scratch);
  p.status = reinterpret_cast<unsigned int*>(p.scratch + tp_tc32_status_offset());
  p.save = reinterpret_cast<uint8_t*>(save); p.n_save = n_save; p.enc_slot = save ? enc_slot : -1;
  const size_t images_per_slot = split_save ? 2 : 1;
  p.save_bits = save ? reinterpret_cast<uint32_t*>(p.save + (size_t)((S + 127) / 128) * n_save * images_per_slot * tc::kABytes) : nullptr;
  void (*kern)(const tcs::Params) = split_save ? tcs::nerf_forward_split_save_kernel
                                    : precision ? tcs::nerf_forward_split_kernel<true> : tcs::nerf_forward_split_kernel<false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tcs::kSmemBytes);
  if (e != cudaSuccess) return (int)e;
  kern<<<grid, tcs::kThreads, tcs::kSmemBytes, (cudaStream_t)stream>>>(p);
  return tp_launch_status();
}

TP_API int tp_tc32_forward(const float* center, const float* ray, const float* depth, int64_t S, int N, int64_t per_image,
                           const void* image, int n_slots, const int32_t* stages, int n_stages, const float* bias,
                           const float* raybias, const float* imgbias, float* rgb, float* density, float* uncert,
                           void* scratch, int64_t scratch_bytes, int precision, void* save, int n_save, int enc_slot, void* stream) {
  if (!center || !ray || !depth || !image || !stages || !bias || !rgb || !density || !uncert || !scratch) return TP_ERR_BAD_ARG;
  if (S < 0 || N < 1 || per_image < 1 || n_stages < 1 || n_stages > tcs::kMaxStages) return TP_ERR_BAD_SHAPE;
  if ((precision != 0 && precision != 1) || (save && (precision != 1 || n_save < 1)) || ((uintptr_t)save & 15)) return TP_ERR_BAD_ARG;
  return tc32_forward_launch(center, ray, depth, S, N, per_image, image, n_slots, stages, n_stages, bias, raybias, imgbias, rgb,
                             density, uncert, scratch, scratch_bytes, precision, save, n_save, enc_slot, false, stream);
}

TP_API int tp_tc32_forward_split_save(const float* center, const float* ray, const float* depth, int64_t S, int N,
                                      int64_t per_image, const void* image, int n_slots, const int32_t* stages, int n_stages,
                                      const float* bias, const float* raybias, const float* imgbias, float* rgb, float* density,
                                      float* uncert, void* scratch, int64_t scratch_bytes, void* save, int n_save, int enc_slot,
                                      void* stream) {
  if (!center || !ray || !depth || !image || !stages || !bias || !rgb || !density || !uncert || !scratch || !save) return TP_ERR_BAD_ARG;
  if (S < 0 || N < 1 || per_image < 1 || n_stages < 1 || n_stages > tcs::kMaxStages || n_save < 1) return TP_ERR_BAD_SHAPE;
  if ((uintptr_t)save & 15) return TP_ERR_ALIGN;
  return tc32_forward_launch(center, ray, depth, S, N, per_image, image, n_slots, stages, n_stages, bias, raybias, imgbias, rgb,
                             density, uncert, scratch, scratch_bytes, 0, save, n_save, enc_slot, true, stream);
}

/* scratch of the render launch: tp_tc32_forward's (parked features, status word), then 256 B, then the view-bias rows */
TP_API int64_t tp_tc32_render_scratch_bytes(void) {
  return tp_tc32_status_offset() + 256 + (int64_t)tp_num_sms() * 8 * tcs::kViewRowFloats * 4;
}

TP_API int tp_tc32_render_forward(const float* kinv, const float* pose_inv, int B, int H, int W, float pix_offset,
                                  const int64_t* ray_idx, int64_t R, int64_t ray0, const float* z_near, const float* z_far, int N,
                                  int depth_mode, const float* rand, uint64_t seed, const void* image, int n_slots,
                                  const int32_t* stages, int n_stages, const float* bias, const float* wview, int L_view,
                                  const float* imgbias_rgb, const float* imgbias, int chains, float min_uncert, float* rgb,
                                  float* rgb_static, float* rgb_transient, float* depth, float* opacity, float* opacity_static,
                                  float* opacity_transient, float* uncert, float* alpha_static, float* alpha_transient,
                                  float* density, void* scratch, int64_t scratch_bytes, int precision, void* stream) {
  if (!kinv || !pose_inv || !z_near || !z_far || !image || !stages || !bias || !wview || !imgbias_rgb || !scratch)
    return TP_ERR_BAD_ARG;
  if (B < 1 || H < 1 || W < 1 || R < 0 || L_view < 0 || L_view > 4 || n_stages < 1 || n_stages > tcs::kMaxStages)
    return TP_ERR_BAD_SHAPE;
  if (N != 32 && N != 64 && N != 128) return TP_ERR_BAD_SHAPE;      // a 128-row tile holds whole rays
  if (!ray_idx && (ray0 < 0 || ray0 + R > (int64_t)H * W)) return TP_ERR_BAD_SHAPE;
  if (depth_mode < 0 || depth_mode > 2 || (depth_mode == 0 && !rand)) return TP_ERR_BAD_ARG;
  if ((precision != 0 && precision != 1) || (chains != 1 && chains != 3)) return TP_ERR_BAD_ARG;
  if (chains == 1 && (rgb_static || rgb_transient || opacity_static || opacity_transient || uncert || alpha_static || alpha_transient))
    return TP_ERR_BAD_ARG;      // the plain model has one chain: rgb, depth, opacity and the per-sample density
  if (((uintptr_t)image & 15) || ((uintptr_t)scratch & 15) || ((uintptr_t)bias & 15) || ((uintptr_t)wview & 15) ||
      ((uintptr_t)imgbias_rgb & 15) || ((uintptr_t)imgbias & 15) || ((uintptr_t)density & (chains == 1 ? 3 : 7)))
    return TP_ERR_ALIGN;
  if (!tp_device_is_sm100()) return TP_ERR_ARCH;
  tcs::RenderParams p = {};
  const int err = tc32_parse_stages(p, stages, n_stages, n_slots, true, imgbias != nullptr, nullptr, 0, -1);
  if (err != TP_OK) return err;
  const int64_t S = (int64_t)B * R * N;
  if (S == 0) return TP_OK;
  if (scratch_bytes < tp_tc32_render_scratch_bytes()) return TP_ERR_WORKSPACE;
  const long long n_tiles = (S + 127) / 128;
  int grid = tp_num_sms();
  if (n_tiles < grid) grid = (int)n_tiles;
  p.S = S; p.N = N; p.per_image = R * N;
  p.image = reinterpret_cast<const uint8_t*>(image); p.bias = bias; p.imgbias = imgbias;
  p.scratch = reinterpret_cast<uint8_t*>(scratch);
  p.status = reinterpret_cast<unsigned int*>(p.scratch + tp_tc32_status_offset());
  p.enc_slot = -1;
  p.kinv = kinv; p.pinv = pose_inv; p.H = H; p.W = W; p.pix_offset = pix_offset;
  p.ray_idx = reinterpret_cast<const long long*>(ray_idx); p.R = R; p.ray0 = ray0;
  p.z_near = z_near; p.z_far = z_far; p.depth_mode = depth_mode; p.rand = rand; p.seed = seed;
  p.wview = wview; p.L_view = L_view; p.imgbias_rgb = imgbias_rgb; p.chains = chains; p.min_uncert = min_uncert;
  p.o_rgb = rgb; p.o_rgb_s = rgb_static; p.o_rgb_t = rgb_transient; p.o_depth = depth; p.o_op = opacity;
  p.o_op_s = opacity_static; p.o_op_t = opacity_transient; p.o_unc = uncert; p.o_as = alpha_static; p.o_at = alpha_transient;
  p.o_density = density;
  p.vrow_off = tp_tc32_status_offset() + 256;
  void (*kern)(const tcs::RenderParams) = precision ? tcs::nerf_render_split_kernel<true> : tcs::nerf_render_split_kernel<false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tcs::kSmemRender);
  if (e != cudaSuccess) return (int)e;
  kern<<<grid, tcs::kThreads, tcs::kSmemRender, (cudaStream_t)stream>>>(p);
  return tp_launch_status();
}

/* The same launch over an object-pixel list: one CTA per SM (the host does not know the list's length); rank shard_rank of
 * shard_world renders its share of the list's super-tiles. */
TP_API int tp_tc32_render_forward_list(const float* kinv, const float* pose_inv, int B, int H, int W, float pix_offset,
                                       const int64_t* list, const int64_t* n_slots, int shard_rank, int shard_world,
                                       const float* z_near, const float* z_far, int N, int depth_mode, const float* rand, uint64_t seed,
                                       const void* image, int n_weight_slots, const int32_t* stages, int n_stages, const float* bias,
                                       const float* wview, int L_view, const float* imgbias_rgb, const float* imgbias, int chains,
                                       float min_uncert, float* rgb, float* rgb_static, float* rgb_transient, float* depth,
                                       float* opacity, float* opacity_static, float* opacity_transient, float* uncert,
                                       float* alpha_static, float* alpha_transient, float* density, void* scratch,
                                       int64_t scratch_bytes, int precision, void* stream) {
  if (!kinv || !pose_inv || !list || !n_slots || !z_near || !z_far || !image || !stages || !bias || !wview || !imgbias_rgb || !scratch)
    return TP_ERR_BAD_ARG;
  if (B < 1 || H < 1 || W < 1 || L_view < 0 || L_view > 4 || n_stages < 1 || n_stages > tcs::kMaxStages) return TP_ERR_BAD_SHAPE;
  if (N != 32 && N != 64 && N != 128) return TP_ERR_BAD_SHAPE;
  if (depth_mode < 0 || depth_mode > 2 || (depth_mode == 0 && !rand)) return TP_ERR_BAD_ARG;      // rand: [B*H*W*N], frame-sized
  if (shard_world < 1 || shard_rank < 0 || shard_rank >= shard_world) return TP_ERR_BAD_ARG;
  if ((precision != 0 && precision != 1) || chains != 3) return TP_ERR_BAD_ARG;      // the static / transient / light model
  if (((uintptr_t)image & 15) || ((uintptr_t)scratch & 15) || ((uintptr_t)bias & 15) || ((uintptr_t)wview & 15) ||
      ((uintptr_t)imgbias_rgb & 15) || ((uintptr_t)imgbias & 15) || ((uintptr_t)density & 7))
    return TP_ERR_ALIGN;
  if (!tp_device_is_sm100()) return TP_ERR_ARCH;
  tcs::ListRenderParams p = {};
  const int err = tc32_parse_stages(p, stages, n_stages, n_weight_slots, true, imgbias != nullptr, nullptr, 0, -1);
  if (err != TP_OK) return err;
  if (scratch_bytes < tp_tc32_render_scratch_bytes()) return TP_ERR_WORKSPACE;
  const int grid = tp_num_sms();
  p.S = 0; p.N = N; p.per_image = (int64_t)H * W * N;      // (list mode takes its rays and its length from the list)
  p.image = reinterpret_cast<const uint8_t*>(image); p.bias = bias; p.imgbias = imgbias;
  p.scratch = reinterpret_cast<uint8_t*>(scratch);
  p.status = reinterpret_cast<unsigned int*>(p.scratch + tp_tc32_status_offset());
  p.enc_slot = -1;
  p.kinv = kinv; p.pinv = pose_inv; p.H = H; p.W = W; p.pix_offset = pix_offset;
  p.z_near = z_near; p.z_far = z_far; p.depth_mode = depth_mode; p.rand = rand; p.seed = seed;
  p.wview = wview; p.L_view = L_view; p.imgbias_rgb = imgbias_rgb; p.chains = chains; p.min_uncert = min_uncert;
  p.o_rgb = rgb; p.o_rgb_s = rgb_static; p.o_rgb_t = rgb_transient; p.o_depth = depth; p.o_op = opacity;
  p.o_op_s = opacity_static; p.o_op_t = opacity_transient; p.o_unc = uncert; p.o_as = alpha_static; p.o_at = alpha_transient;
  p.o_density = density;
  p.vrow_off = tp_tc32_status_offset() + 256;
  p.list = reinterpret_cast<const long long*>(list); p.n_slots = reinterpret_cast<const long long*>(n_slots);
  p.shard_rank = shard_rank; p.shard_world = shard_world;
  void (*kern)(const tcs::ListRenderParams) = precision ? tcs::nerf_render_list_split_kernel<true> : tcs::nerf_render_list_split_kernel<false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tcs::kSmemRender);
  if (e != cudaSuccess) return (int)e;
  kern<<<grid, tcs::kThreads, tcs::kSmemRender, (cudaStream_t)stream>>>(p);
  return tp_launch_status();
}
