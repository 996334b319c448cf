// Stage table, kernel parameters and the per-sample encoder of the fused forward kernel (mlp_tc.cu: two lock-stepped tiles
// per CTA) and its accumulator-drain helpers (mlp_tc_epilogue.cuh).
#pragma once
#include "tc_common.cuh"
#include "rays.cuh"

namespace tc {

constexpr uint32_t kEBytes = 16384;    // 128 x 64 bf16 encoding tile
constexpr int kNumLayers = 17;
constexpr int kNumChunks = 122;

// stage table: chunks read from A (K=32 each), chunks read from E, small (N=16, one chunk spans K=256),
// kind of epilogue, bias handling, needs the feature reload first.
// Static biases of the 256-wide stages ride on the tensor cores: column 63 of the encoding tile is a constant 1 and
// the bias sits in the matching weight column -- for stages that read E anyway (trunk 0 and 4) inside their last E
// chunk, for the others as one extra K=16 step on E columns 48..63 with an 8 KB weight chunk that is zero except for
// that column (BIAS_MMA).  Their epilogue is then a pure convert.  Per-ray / per-image biases (fp32 tables) and the
// three N=16 output stages add their bias in the epilogue.
// The N=16 output stages carry their weight rows TWICE: rows 0..7 = bf16(W), rows 8..15 = bf16(W - bf16(W)) -- the epilogue
// adds column c and column c + 8, so the output layers see ~16 mantissa bits of their weights at no extra MMA (the systematic
// rounding of these few rows was the largest term of the bf16 gradient error: DESIGN.md section 2).
enum Epi : int { EPI_HIDDEN = 0, EPI_DENSITY = 1, EPI_RGB_OUT = 2, EPI_TRANS_OUT = 3 };
enum BiasKind : int { BIAS_MMA = 0, BIAS_RAY = 1, BIAS_IMAGE = 2, BIAS_SMALL = 3 };
struct Layer {
  int a_chunks, e_chunks, small, epi, bias_kind, bias_chunk, reload;
};
static __constant__ Layer kLayers[kNumLayers] = {
    {0, 2, 0, EPI_HIDDEN, BIAS_MMA, 0, 0},       // trunk 0  (63 -> 256); bias in E column 63 of its own chunk
    {8, 0, 0, EPI_HIDDEN, BIAS_MMA, 1, 0},       // trunk 1
    {8, 0, 0, EPI_HIDDEN, BIAS_MMA, 1, 0},       // trunk 2
    {8, 0, 0, EPI_HIDDEN, BIAS_MMA, 1, 0},       // trunk 3
    {8, 2, 0, EPI_HIDDEN, BIAS_MMA, 0, 0},       // trunk 4  (skip: [feat | enc]); bias in E column 63
    {8, 0, 0, EPI_HIDDEN, BIAS_MMA, 1, 0},       // trunk 5
    {8, 0, 0, EPI_HIDDEN, BIAS_MMA, 1, 0},       // trunk 6
    {8, 0, 1, EPI_DENSITY, BIAS_SMALL, 0, 0},    // trunk 7 row 0     -> sigma_static (softplus)
    {8, 0, 0, EPI_HIDDEN, BIAS_MMA, 1, 0},       // trunk 7 rows 1..  -> feature (relu); parked to L2 afterwards
    {8, 1, 0, EPI_HIDDEN, BIAS_RAY, 0, 0},       // rgb 0    ([feat | xyz]; view+light folded into the ray bias)
    {8, 0, 0, EPI_HIDDEN, BIAS_MMA, 1, 0},       // rgb 1
    {8, 0, 0, EPI_HIDDEN, BIAS_MMA, 1, 0},       // rgb 2
    {8, 0, 1, EPI_RGB_OUT, BIAS_SMALL, 0, 0},    // rgb 3    -> sigmoid
    {8, 0, 0, EPI_HIDDEN, BIAS_IMAGE, 0, 1},     // trans 0  (feature reloaded; transient latent in the image bias)
    {8, 0, 0, EPI_HIDDEN, BIAS_MMA, 1, 0},       // trans 1
    {8, 0, 0, EPI_HIDDEN, BIAS_MMA, 1, 0},       // trans 2
    {8, 0, 1, EPI_TRANS_OUT, BIAS_SMALL, 0, 0}   // trans 3  -> sigmoid x3, softplus x2
};
constexpr int kSpillLayer = 8, kReloadIssueLayer = 12;
constexpr int kStaticLayers = 13;      // stages 0..12: trunk, density, feature, rgb head
constexpr int kSaveSlots = 7;
// activation-save slot of each stage (training): feat, rgb h1..h3, trans h1..h3; -1 = not saved
static __constant__ int kSaveSlot[kNumLayers] = {-1, -1, -1, -1, -1, -1, -1, -1, 0, 1, 2, 3, -1, 4, 5, 6, -1};
// ReLU-bitmask slot of each stage (training): rgb h1, h2, trans h1, h2 -> 0..3 ([8 word planes][128 rows] = 4 KB per tile and slot,
// stored behind the tile images of the save buffer); the backward chain reads these instead of the 64 KB activation tiles
static __constant__ int kMaskBitSlot[kNumLayers] = {-1, -1, -1, -1, -1, -1, -1, -1, -1, 0, 1, -1, -1, 2, 3, -1, -1};
constexpr int kMaskBitSlots = 4;
constexpr uint32_t kMaskBitBytes = 4096;
constexpr int kSmallBiasOffset = 0;            // biasbuf: [density b, rgb3 b(3), trans3 b(5)] (fp32, 16 floats)

struct Params {
  // list mode of the render launch (kMode 4, tp_render_fused_forward_list) keeps its inputs in the slots of per-sample inputs it
  // does not read: the layout, and with it the code of every other launch, is that of the plain struct
  union {
    const float* center;     // [rays,3]                              (per-sample launches; the render launch generates rays)
    const long long* list;   // list mode: object-pixel list (tp_mask_ray_list), entry q = view * HW + pixel, pad ~(view * HW)
  };
  union {
    const float* ray;        // [rays,3]
    const long long* n_slots;      // list mode: DEVICE count of list entries (a multiple of 256 / N)
  };
  union {
    const float* depth;      // [S]
    struct { int shard_rank, shard_world; };      // list mode: this rank renders super-tiles [r T / w, (r + 1) T / w)
  };
  long long S;
  int N;                     // samples per ray
  long long per_image;       // samples per image
  const uint8_t* packed;     // kNumChunks x 16 KB weight image
  const float* biasbuf;      // 16 floats: biases of the three N=16 output stages
  const float* raybias;      // [rays,256]  rgb-0 bias incl. view encoding + light latent (per-sample launches)
  const float* imgbias;      // [images,256] trans-0 bias incl. transient latent
  float* rgb;                // [S,3,2]
  float* density;            // [S,2]
  float* uncert;             // [S]
  uint8_t* scratch;          // gridDim.x x 2 x 64 KB (parked features)
  uint8_t* bits;             // optional [tiles][4][8 planes][128 rows] ReLU bitmask words (training; lives behind `save`)
  uint8_t* save;             // optional [tiles][7][64 KB]: feat, rgb h1..h3, trans h1..h3 tile images for the backward
  long long prof_offset;     // byte offset of the cycle counters inside `scratch` (-DTP_FWD_PROF builds only)
  int n_layers;              // 17 = all stages; 13 = static only (rendering that needs neither the transient head nor uncert):
                             // the stage list stops after the rgb output, transient outputs are written as zeros.  Host side only:
                             // it selects the kernel instantiation (the kernel takes the count as a template parameter)
  // ---- fused render launch (mode 3, tp_render_fused_forward): rays, sample depths, the view-direction bias and the
  // compositing all happen in the kernel; per ray it reads 8 B (+ 8 B of ray index) and writes 56 B
  const float* kinv;         // [B,9]  K^-1 per view (camera.py:292-314; host-side inverses as in the reference)
  const float* pinv;         // [B,12] pose^-1 per view
  int H, W;
  float pix_offset;          // 0.5 (camera.py:301-302)
  const long long* ray_idx;  // [B,R] pixel index of each ray, or NULL: ray r of a view is pixel ray0 + r
  long long R, ray0;
  const float* z_near;       // [B,H*W] full-frame sample bounds (data/lm.py:316-365), read at the ray's pixel
  const float* z_far;
  const float* rand;         // [S] injected stratified jitter (depth_mode 0), else NULL
  int depth_mode;            // 0 = injected rand, 1 = midpoints, 2 = in-kernel Philox (same stream as tp_sample_depth)
  unsigned long long seed;
  const float* wview;        // [3+6L][256] fp32: columns 256.. of mlp_rgb[0].weight, transposed (view-direction inputs)
  int L_view;
  const float* imgbias_rgb;  // [B,256] rgb-0 bias + light-latent part (tp_tc_image_biases)
  float min_uncert;
  float* o_rgb;              // per-ray outputs (any may be NULL): [B*R,3] x 3, [B*R] x 5
  float* o_rgb_s;
  float* o_rgb_t;
  float* o_depth;
  float* o_op;
  float* o_op_s;
  float* o_op_t;
  float* o_unc;
  float* o_as;               // per-sample outputs (any may be NULL): alpha_static [S], alpha_transient [S]; `density` [S,2]
  float* o_at;
};

// positional encoding of one point as the 32 packed bf16x2 words of its E-tile row: [x,y,z, per coord sin(2^k pi x) k<10,
// cos(...) k<10, 1].  sincospif gives the exact-argument octave 0; higher octaves by the double-angle recurrence (error <<
// bf16 ulp).  Kept in registers so the arithmetic can run while the E tile is still being read by the previous super-tile.
__device__ __forceinline__ void encode_xyz_regs(const float (&xyz)[3], uint32_t (&e)[32]) {
  float v[64];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const float x = xyz[j];
    v[j] = x;
    float sn, cs;
    sincospif(x, &sn, &cs);
#pragma unroll
    for (int k = 0; k < 10; ++k) {
      v[3 + j * 20 + k] = sn;
      v[3 + j * 20 + 10 + k] = cs;
      const float s2 = 2.f * sn * cs, c2 = (cs - sn) * (cs + sn);
      sn = s2;
      cs = c2;
    }
  }
  v[63] = 1.f;   // constant-1 column: carries the static biases through the MMA
#pragma unroll
  for (int i = 0; i < 32; ++i) e[i] = pack_bf16(v[2 * i], v[2 * i + 1]);
}
__device__ __forceinline__ void encode_regs(const float (&c)[3], const float (&r)[3], float d, uint32_t (&e)[32]) {
  const float xyz[3] = {__fadd_rn(c[0], __fmul_rn(r[0], d)), __fadd_rn(c[1], __fmul_rn(r[1], d)), __fadd_rn(c[2], __fmul_rn(r[2], d))};
  encode_xyz_regs(xyz, e);      // x = c + ray * d (camera.py:317-322), one rounding per operation
}
__device__ __forceinline__ void store_encoding(const uint32_t (&e)[32], uint32_t e_smem, int row) {
#pragma unroll
  for (int k8 = 0; k8 < 8; ++k8) st_shared_v4(e_smem + k8 * 2048 + row * 16, e[4 * k8], e[4 * k8 + 1], e[4 * k8 + 2], e[4 * k8 + 3]);
}
__device__ __forceinline__ void encode_point(const float (&c)[3], const float (&r)[3], float d, uint32_t e_smem, int row) {
  uint32_t e[32];
  encode_regs(c, r, d, e);
  store_encoding(e, e_smem, row);
}

__device__ __forceinline__ void encode_sample(const Params& p, long long s, uint32_t e_smem, int row) {
  const long long r = s / p.N;
  const float c[3] = {p.center[r * 3], p.center[r * 3 + 1], p.center[r * 3 + 2]};
  const float ry[3] = {p.ray[r * 3], p.ray[r * 3 + 1], p.ray[r * 3 + 2]};
  encode_point(c, ry, p.depth[s], e_smem, row);
}

}  // namespace tc
