// Implicit-GEMM convolution on the 5th-gen tensor cores (tcgen05 + TMEM), operands staged by TMA.
//
// One kernel family covers every dense layer of the hot path (1x1x1, causal (2,3,3) / (1,3,3) 3-D, dilated 3x3,
// 7x7 stride 2, 3x3 / 1x1 stride 2): a convolution is a sum over taps of [pixels x Cin] . [Cin x Cout] GEMMs whose
// A operand is a shifted (strided, zero-padded) window of the channels-last activation tensor -- exactly what a
// 5-D TMA box with out-of-bounds zero fill delivers.
//
// Precision: fp32 tensors are carried as two bf16 planes (hi = bf16(x), lo = bf16(x - hi)); every product is
// evaluated as hi*hi + hi*lo + lo*hi on the bf16 tensor pipe with fp32 accumulation in TMEM (error ~2^-16 per
// product instead of 2^-8), which keeps 25 stacked layers inside the 1e-3 parity bar.  Eval-mode BatchNorm is
// folded into the weights/bias on the host; bias, per-image bias (pyramid-pool / ASPP-pool / ego-motion
// branches), ReLU, residual add and the concat offset are fused in the epilogue.
//
//   tile     : 256 output pixels (16 x 16 of one image = two UMMA M=128 sub-tiles sharing every weight tile) x BN
//              output channels (64 / 128; 256 runs as two launches)
//   K loop   : taps x (Cin / 64); TMA brings A_hi, A_lo (256 or 288 pixel rows x 64 bf16, 128B-swizzled; one load
//              serves the three dy taps of a 3x3) and B_hi, B_lo (BN x 64; small weight tensors stay resident in
//              smem) through separate rings; one thread issues 2 x 4 (UMMA_K=16) x 3 tcgen05.mma per tap
//   CTA      : persistent, one per SM, walks tiles blockIdx.x + i*gridDim.x
//   warps    : 0 = TMA producer, 1 = MMA issuer + TMEM allocator, 2..9 = epilogue (TMEM -> regs -> global), which
//              drains one accumulator pair while the tensor pipe fills the other
//
// Reference layers: stp3/layers/temporal.py:252-489, stp3/layers/convolutions.py:183-280, stp3/models/decoder.py.
#include <cuda_bf16.h>

#include <cstdlib>

#include "common.cuh"
#include "ptx.cuh"

namespace stp3 {

constexpr int kEpiWarps = 8;                     // two warps per TMEM lane quarter, each owning half of the columns
constexpr int kConvThreads = 64 + kEpiWarps * 32;
constexpr int kSubH = 8, kTileW = 16;           // one UMMA M=128 sub-tile = 8 x 16 pixels; a tile stacks n_sub (1 or 2) of them
constexpr int kBK = 64;                         // channels per K step (one 128-byte swizzle row of bf16)
constexpr int kMaxTaps = 49;
constexpr int kMaxAStages = 4, kMaxBStages = 8;
constexpr int kMaxHeadOut = 8;

struct ConvParams {
  int n_img, T, t0, Ho, Wo;
  int T_total;              // frames of the input tensor
  int H, W;                 // input image size
  int skip_t;               // skip tap groups whose window lies entirely in the zero padding for the whole tile (frame
                            // outside [0, T_total): causal convs at t = 0; rows / columns outside the image: dilated convs)
  int tiles_x, tiles_y, n_tiles;
  int stride;
  int kblocks;              // Cin / 64 of this convolution
  int cin_off;              // first input channel inside the (wider) input tensor, multiple of 64
  int ntaps;
  int ks_first, ks_end;     // UMMA_K = 16 steps that carry data: [ks_first, 4) of the first K block, [0, ks_end) of the last
                            // (channels outside are zero padding of a narrow convolution: neither multiplied nor needed)
  int n_sub;                // sub-tiles per tile: 2 (16x16 pixels, weight tiles shared) or 1 (small images: more tiles)
  // taps that share one activation load: consecutive taps with the same (dt, dx) whose dy advance by the stride read
  // the same strided rows shifted by one OUTPUT row each (the three dy taps of a 3x3; dy = -3,-1,1,3 / -2,0,2 of the
  // stride-2 7x7), so one box of tile_rows + gmax - 1 rows serves the whole group
  int n_groups, gmax;
  unsigned char gstart[kMaxTaps], gsize[kMaxTaps];
  int a_plane_bytes;        // bytes of one activation plane of a stage = box_h * 16 px * 128 B
  int n_mma;                // output columns the MMAs compute (multiple of 16, <= BN): columns beyond the convolution's
                            // real Cout have zero weights and bias, so they are neither loaded nor multiplied
  int b_rows;               // weight rows of one plane part held by this CTA: n_mma, or n_mma / 2 in a pair
  int b_tile_bytes;         // shared-memory bytes of one K step's weights (2 parts; 3 for a stacked pair)
  int w_rows;               // rows per (tap, kb, plane) block of the packed weight tensor (the convolution's padded Cout)
  int w_row_off;            // first row of this launch inside that block (a 256-channel conv runs as two launches)
  signed char tap[kMaxTaps][4];   // (dt, dy, dx): input coordinate = output coordinate * stride + d
  const float* bias;        // [BN]
  const float* img_bias;    // [n_img][img_bias_stride] or null (replaces bias)
  int img_bias_stride;
  int relu;
  int res_mode;             // 0 none, 1 residual added before the activation, 2 after
  const __nv_bfloat16* res_hi;
  const __nv_bfloat16* res_lo;
  int res_cstride, res_coff;
  __nv_bfloat16* out_hi;    // channels-last (n_img, Ho, Wo, out_cstride), may be null when out_f32 is used
  __nv_bfloat16* out_lo;
  int out_cstride, out_coff, n_store;
  int vec256;               // bit 0: output rows / windows are 32-byte aligned (256-bit stores), bit 1: residual likewise
  float* out_f32;           // optional (n_img, n_valid, Ho, Wo) fp32, the reference's NCHW layout
  int n_valid, f32_coff;    // channel offset of this launch inside out_f32
  int f32_nhwc;             // out_f32 is channels-last (n_img, Ho, Wo, n_valid): 16 channels of a pixel = two 32-byte stores
  int sigmoid;              // apply to out_f32 (instance_center head)
  int na_stages, nb_stages; // smem ring depths chosen by the host
  int b_resident;           // all weight tiles of the convolution stay in shared memory for the CTA's lifetime
  // fused 1x1 "head" on the activated tile: out_k = head_b[k] + sum_c head_w[k][c] * y[c]  (decoder heads 3x3 -> 1x1)
  int head_ko;              // 0 = off, else 1..8 outputs
  const float* head_w;      // [head_ko][BN]
  const float* head_b;      // [head_ko]
  float* head_out[8];       // plane of output k for image 0 (fp32, (Ho, Wo))
  long long head_img_stride[8];   // elements between consecutive images for output k
  int head_sigmoid_mask;    // bit k: sigmoid on output k
  // second destination (BN = 128): output columns [64, 128) go to another tensor with their own activation flag -- two
  // 64-column convolutions that read the same input run as one launch and read it once
  __nv_bfloat16* out2_hi;
  __nv_bfloat16* out2_lo;
  int out2_cstride, out2_coff, n_store2, relu2;
  // per-image column sums of the activated output (the consumer's pooling branches need sum over H*W): every epilogue
  // warp keeps running sums of its pixels in registers and writes one partial row per (CTA, lane quarter, image) --
  // plain stores, fixed order: deterministic.  BN = 64 only.  sum_part: [gridDim.x][4][n_img][BN], zeroed by the host.
  float* sum_part;
  // linear tiling (LINEAR = true): a tile is 128 (256 for a pair) consecutive output pixels of the flattened
  // (image, oy, ox) space; one im2col TMA load per (tap, K block) brings them, zero-filled outside the image
  int m_total;              // n_img * Ho * Wo
  int lin_lo_w, lin_lo_h;   // lower corner of the im2col bounding box (smallest tap offset); a tap loads at d - lo
  // work units: (tile, column half); n_halves = 2 runs a 256-column convolution in one launch (linear tiling only)
  int n_halves, n_units;
};

// STACK (BN = 64 only): the hi and lo weight planes of a K step form ONE B operand of 2*BN rows, so a product is two
// MMAs instead of three -- A_hi x [W_hi; W_lo] (N = 2*BN) and A_lo x W_hi (N = BN) -- and the activation tile is read
// from shared memory twice instead of three times (N = 64 MMAs are bound by exactly those reads).  The accumulator
// has 2*BN columns; the epilogue adds columns c and BN + c.
template <int BN, bool PAIR = false, bool STACK = false, bool LINEAR = false>
struct ConvSmem {
  static constexpr int kBRows = PAIR ? BN / 2 : BN;                    // weight rows held by one CTA (a pair splits N)
  // B_hi + B_lo of one K step; a stacked pair holds [own half of the stacked operand (BN rows)][own half of W_hi]
  static constexpr int kBTileBytes = (STACK && PAIR ? 3 : 2) * kBRows * kBK * 2;
  static constexpr int kAccCols = STACK ? 2 * BN : BN;                 // TMEM columns of one accumulator
  static constexpr int kTmemCols = 4 * kAccCols;                       // 2 sub-tiles x 2 accumulator buffers
  static constexpr int kBiasCols = LINEAR ? 2 * BN : BN;               // bias of both column halves
  static constexpr size_t tail_bytes() {
    return (kBiasCols + kMaxHeadOut * BN) * sizeof(float) + kMaxHeadOut * 128 * sizeof(float) + kEpiWarps * 64 * sizeof(float) +
           (2 * kMaxAStages + 2 * kMaxBStages + 8) * 8;
  }
};

// true if every input element the tap group touches for this tile is zero padding (same answer in the producer and
// the MMA issuer, and in both CTAs of a pair: it looks at the whole tile)
__device__ __forceinline__ bool group_is_padding(const ConvParams& p, int grp, int tidx, int oy_tile, int ox0, int tile_h) {
  const int tap0 = p.gstart[grp];
  const int t = tidx + p.tap[tap0][0];
  const int ylo = oy_tile * p.stride + p.tap[tap0][1];
  const int yhi = (oy_tile + tile_h - 1 + p.gsize[grp] - 1) * p.stride + p.tap[tap0][1];
  const int xlo = ox0 * p.stride + p.tap[tap0][2];
  const int xhi = (ox0 + kTileW - 1) * p.stride + p.tap[tap0][2];
  return t < 0 || t >= p.T_total || yhi < 0 || ylo >= p.H || xhi < 0 || xlo >= p.W;
}

// Persistent, warp-specialised implicit-GEMM convolution.
//   * A CTA walks output tiles blockIdx.x + i*gridDim.x; a tile is 16x16 pixels = two M=128 sub-tiles that share every
//     weight tile (B traffic per flop halves).
//   * Activations and weights travel through separate shared-memory rings.  For 3x3 / stride 1 / dilation 1 kernels one
//     activation load of 18 image rows serves the three dy taps: their A operands are the same smem tile at row
//     offsets 0, 16, 32 (2 KB steps keep the 1024-byte swizzle alignment), so A traffic drops 2.4x.
//   * The MMA thread alternates between two TMEM accumulator buffers; eight epilogue warps drain one while the tensor
//     pipe fills the other.
//
// PAIR = true: two CTAs of a cluster (one TPC) share a 16x16 tile through tcgen05.mma.cta_group::2 (UMMA M = 256): each
// CTA stages its own 8 image rows of A and HALF of the weight rows, the leader (cluster rank 0) issues every MMA, both
// tensor cores read both weight halves, and each CTA's epilogue drains its own 128 accumulator rows.  Shared-memory
// operand reads per MMA drop by a quarter and the weight traffic per SM halves.  Barrier protocol: "full" barriers
// live in the leader and collect the TMA bytes of both CTAs; "empty" / "accumulator ready" are multicast commits;
// "accumulator drained" collects the epilogue warps of both CTAs in the leader.
//
// LINEAR = true: a tile is 128 consecutive output pixels of the flattened (image, oy, ox) space per CTA (256 for a
// pair; n_sub = 1), so rows and images are crossed and only the tail of the last tile is wasted -- small maps (50^2,
// 25^2) otherwise compute up to 39 % padding pixels in 16x16 tiles.  tm_a_hi / tm_a_lo are rank-4 im2col maps; every
// (tap, K block) is its own A load (no dy sharing), issued in the same (group, K block, tap) order as the 2-D tiling
// so each pixel accumulates the same products in the same order.  A work unit is (tile, column half): a 256-column
// convolution walks both halves in one launch.
template <int BN, bool PAIR, bool STACK, bool LINEAR>
__global__ void __launch_bounds__(kConvThreads, 1)
conv_igemm_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                  const __grid_constant__ CUtensorMap tm_w, const ConvParams p) {
  using S = ConvSmem<BN, PAIR, STACK, LINEAR>;
  constexpr int kLinTile = PAIR ? 256 : 128;      // output pixels of a linear tile
  static_assert(!STACK || BN == 64, "stacked weight operand: BN = 64 only (TMEM columns)");
  const int kBRows = p.b_rows;
  const uint32_t rank = PAIR ? ptx::cluster_ctarank() : 0u;              // 0 = leader
  const int cta = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;       // tile walker id (a pair walks together)
  const int n_cta = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  constexpr uint32_t kProd = PAIR ? 2 : 1;                               // producers arriving on a "full" barrier
  extern __shared__ unsigned char smem_raw[];
  // 1024-byte alignment for the 128-byte swizzle; plain offset arithmetic keeps the pointer in the shared state space
  unsigned char* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  const int k_iters = p.ntaps * p.kblocks;
  const bool resident = p.b_resident != 0;
  const int a_stage_bytes = 2 * p.a_plane_bytes;
  unsigned char* a_ring = smem;
  unsigned char* b_ring = a_ring + (size_t)p.na_stages * a_stage_bytes;            // ring, or the resident weights
  float* s_bias = reinterpret_cast<float*>(b_ring + (size_t)(resident ? k_iters : p.nb_stages) * p.b_tile_bytes);
  float* s_head = s_bias + S::kBiasCols;          // [kMaxHeadOut][BN]
  float* s_hx = s_head + kMaxHeadOut * BN;        // [kMaxHeadOut][128] head partials handed between column halves
  float* s_wb = s_hx + kMaxHeadOut * 128;         // [kEpiWarps][64] per-image bias slice of each epilogue warp
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_wb + kEpiWarps * 64);
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + kMaxAStages;
  uint64_t* b_full = a_empty + kMaxAStages;
  uint64_t* b_empty = b_full + kMaxBStages;
  uint64_t* tmem_full_bar = b_empty + kMaxBStages;       // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;          // [2]
  uint64_t* bres_bar = tmem_empty_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bres_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // Programmatic dependent launch: the next conv of the stream may set up (barriers, TMEM, resident weights) on SMs
  // this grid has left; this grid's own set-up ran while its predecessor drained.  Only module constants (bias,
  // weights, head weights) are read before griddep_wait().
  ptx::griddep_launch_dependents();
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tm_a_hi); ptx::prefetch_tmap(&tm_a_lo); ptx::prefetch_tmap(&tm_w);
    for (int i = 0; i < p.na_stages; ++i) { ptx::mbar_init(&a_full[i], kProd); ptx::mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < p.nb_stages; ++i) { ptx::mbar_init(&b_full[i], kProd); ptx::mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&tmem_full_bar[i], 1);
      ptx::mbar_init(&tmem_empty_bar[i], kEpiWarps * kProd);
    }
    ptx::mbar_init(bres_bar, kProd);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    if constexpr (PAIR) ptx::tmem_alloc_pair<S::kTmemCols>(tmem_slot);
    else ptx::tmem_alloc<S::kTmemCols>(tmem_slot);
  }
  for (int i = threadIdx.x; i < BN * p.n_halves; i += blockDim.x) s_bias[i] = p.bias[i];
  for (int i = threadIdx.x; i < p.head_ko * BN; i += blockDim.x) s_head[i] = p.head_w[i];
  ptx::tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) ptx::cluster_sync();        // the peer's barriers are initialised before anyone signals them
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int tiles_per_img = p.tiles_x * p.tiles_y;
  const int n_groups = p.n_groups;
  const int tile_h = PAIR ? 2 * kSubH : kSubH * p.n_sub;      // image rows of a tile (a pair: 8 per CTA)
  const int hw_out = p.Ho * p.Wo;

  if (warp == 0) {
    // ===================== TMA producer (whole warp walks the loops; one elected lane issues) =====================
    {
      // in a pair every "full" barrier is the leader's: arrive / complete_tx go through its shared::cluster address.
      // load_b: the weight tile of K step `it` into `dst` (called by the elected lane; transaction bytes on `bar`)
      int w_row_off = p.w_row_off;                // + BN for the upper column half of a work unit
      auto load_b = [&](unsigned char* dst, int it, uint64_t* bar) {
        const int row_hi = (it * 2) * p.w_rows + w_row_off, row_lo = row_hi + p.w_rows;
        if constexpr (PAIR) {
          const uint32_t cbar = ptx::mapa(ptx::smem_u32(bar), 0);
          if constexpr (STACK) {
            // stacked operand [W_hi; W_lo]: the leader holds W_hi, the peer W_lo; then each its half of W_hi
            const int r0 = rank ? row_lo : row_hi;
            ptx::tma_load_2d_pair(dst, &tm_w, cbar, 0, r0);
            ptx::tma_load_2d_pair(dst + kBRows * kBK * 2, &tm_w, cbar, 0, r0 + kBRows);
            ptx::tma_load_2d_pair(dst + 2 * kBRows * kBK * 2, &tm_w, cbar, 0, row_hi + (int)rank * kBRows);
          } else {
            ptx::tma_load_2d_pair(dst, &tm_w, cbar, 0, row_hi + (int)rank * kBRows);
            ptx::tma_load_2d_pair(dst + kBRows * kBK * 2, &tm_w, cbar, 0, row_lo + (int)rank * kBRows);
          }
        } else {
          ptx::tma_load_2d(dst, &tm_w, bar, 0, row_hi);                       // [W_hi; W_lo], also the stacked operand
          ptx::tma_load_2d(dst + kBRows * kBK * 2, &tm_w, bar, 0, row_lo);
        }
      };
      auto expect_b = [&](uint64_t* bar, uint32_t bytes) {
        if constexpr (PAIR) ptx::mbar_arrive_expect_tx_cluster(ptx::mapa(ptx::smem_u32(bar), 0), bytes);
        else ptx::mbar_arrive_expect_tx(bar, bytes);
      };
      if (resident && ptx::elect_one_sync()) {
        expect_b(bres_bar, (uint32_t)(k_iters * p.b_tile_bytes));
        for (int it = 0; it < k_iters; ++it) load_b(b_ring + (size_t)it * p.b_tile_bytes, it, bres_bar);
      }
      __syncwarp();
      ptx::griddep_wait();                        // activations come from the preceding kernel
      int as = 0, bs = 0; uint32_t aph = 0, bph = 0;
      for (int unit = cta; unit < p.n_units; unit += n_cta) {
        const int tile = LINEAR ? unit / p.n_halves : unit;
        if constexpr (LINEAR) w_row_off = p.w_row_off + (unit % p.n_halves) * BN;
        int img, oy0, ox0;                        // first output pixel this CTA loads
        if constexpr (LINEAR) {
          int m = tile * kLinTile + (int)rank * 128;
          if (m >= p.m_total) m = 0;              // the peer's rows of a last pair tile: loaded, never stored
          img = m / hw_out;
          const int rem = m - img * hw_out;
          oy0 = rem / p.Wo; ox0 = rem - oy0 * p.Wo;
        } else {
          img = tile / tiles_per_img;
          const int rem = tile % tiles_per_img;
          oy0 = (rem / p.tiles_x) * tile_h + (int)rank * kSubH; ox0 = (rem % p.tiles_x) * kTileW;
        }
        const int bidx = img / p.T, tidx = p.t0 + img % p.T;
        for (int grp = 0; grp < n_groups; ++grp) {
          const int tap0 = p.gstart[grp], gsz = p.gsize[grp];
          // linear: the start of the traversal inside the im2col bounding box; the tap travels as the load's offset
          const int x = ox0 * p.stride + (LINEAR ? p.lin_lo_w : p.tap[tap0][2]);
          const int y = oy0 * p.stride + (LINEAR ? p.lin_lo_h : p.tap[tap0][1]);
          const int t = tidx + p.tap[tap0][0];
          if (!LINEAR && p.skip_t && group_is_padding(p, grp, tidx, oy0 - (int)rank * kSubH, ox0, tile_h)) continue;
          // the activation stage of tap group member j (linear: its own im2col load; 2-D: one box for the group)
          auto load_a = [&](int kb, int j) {
            ptx::mbar_wait(&a_empty[as], aph ^ 1);
            if (ptx::elect_one_sync()) {
              unsigned char* sa = a_ring + (size_t)as * a_stage_bytes;
              const int c = p.cin_off + kb * kBK;
              if constexpr (LINEAR) {
                const uint16_t ow = (uint16_t)(p.tap[tap0 + j][2] - p.lin_lo_w);
                const uint16_t oh = (uint16_t)(p.tap[tap0 + j][1] - p.lin_lo_h);
                if constexpr (PAIR) {
                  const uint32_t bar = ptx::mapa(ptx::smem_u32(&a_full[as]), 0);
                  ptx::mbar_arrive_expect_tx_cluster(bar, (uint32_t)a_stage_bytes);
                  ptx::tma_load_im2col_4d_pair(sa, &tm_a_hi, bar, c, x, y, img, ow, oh);
                  ptx::tma_load_im2col_4d_pair(sa + p.a_plane_bytes, &tm_a_lo, bar, c, x, y, img, ow, oh);
                } else {
                  ptx::mbar_arrive_expect_tx(&a_full[as], (uint32_t)a_stage_bytes);
                  ptx::tma_load_im2col_4d(sa, &tm_a_hi, &a_full[as], c, x, y, img, ow, oh);
                  ptx::tma_load_im2col_4d(sa + p.a_plane_bytes, &tm_a_lo, &a_full[as], c, x, y, img, ow, oh);
                }
              } else if constexpr (PAIR) {
                const uint32_t bar = ptx::mapa(ptx::smem_u32(&a_full[as]), 0);
                ptx::mbar_arrive_expect_tx_cluster(bar, (uint32_t)a_stage_bytes);
                ptx::tma_load_5d_pair(sa, &tm_a_hi, bar, c, x, y, t, bidx);
                ptx::tma_load_5d_pair(sa + p.a_plane_bytes, &tm_a_lo, bar, c, x, y, t, bidx);
              } else {
                ptx::mbar_arrive_expect_tx(&a_full[as], (uint32_t)a_stage_bytes);
                ptx::tma_load_5d(sa, &tm_a_hi, &a_full[as], c, x, y, t, bidx);
                ptx::tma_load_5d(sa + p.a_plane_bytes, &tm_a_lo, &a_full[as], c, x, y, t, bidx);
              }
            }
            __syncwarp();
            if (++as == p.na_stages) { as = 0; aph ^= 1; }
          };
          auto load_w = [&](int kb, int j) {
            const int it = (tap0 + j) * p.kblocks + kb;              // [tap][kb][plane][rows] blocks of 64-wide rows
            ptx::mbar_wait(&b_empty[bs], bph ^ 1);
            if (ptx::elect_one_sync()) {
              expect_b(&b_full[bs], (uint32_t)p.b_tile_bytes);
              load_b(b_ring + (size_t)bs * p.b_tile_bytes, it, &b_full[bs]);
            }
            __syncwarp();
            if (++bs == p.nb_stages) { bs = 0; bph ^= 1; }
          };
          for (int kb = 0; kb < p.kblocks; ++kb) {
            if constexpr (LINEAR) {
              for (int j = 0; j < gsz; ++j) {                        // A and W of each tap in turn: the issuer
                load_a(kb, j);                                       // consumes them in this order
                if (!resident) load_w(kb, j);
              }
            } else {
              load_a(kb, 0);
              if (!resident) for (int j = 0; j < gsz; ++j) load_w(kb, j);
            }
          }
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ===================== MMA issuer (whole warp walks the loops; one elected lane issues) =====================
    {
      const uint32_t idesc = ptx::umma_idesc_bf16(PAIR ? 256 : 128, p.n_mma);
      const uint32_t idesc2 = ptx::umma_idesc_bf16(PAIR ? 256 : 128, 2 * p.n_mma);     // stacked operand
      // plain (CTA-scope) waits also for the barriers the peer signals: the data they guard moves through the async
      // proxy (TMA -> UMMA) or TMEM (ordered by the tcgen05 fences); a cluster-scope acquire on the MMA-issuing thread
      // costs ~0.7 us per wait and starves the tensor pipe
      auto wait_full = [](uint64_t* bar, uint32_t ph) { ptx::mbar_wait(bar, ph); };
      auto mma = [](uint32_t d, uint64_t a, uint64_t b, uint32_t id, uint32_t acc) {
        if constexpr (PAIR) ptx::umma_bf16_pair(d, a, b, id, acc); else ptx::umma_bf16(d, a, b, id, acc);
      };
      auto commit = [](uint64_t* bar) {
        if constexpr (PAIR) ptx::umma_commit_pair(bar); else ptx::umma_commit(bar);
      };
      if (resident) wait_full(bres_bar, 0);
      int as = 0, bs = 0; uint32_t aph = 0, bph = 0;
      int buf = 0; uint32_t acc_phase = 0;
      for (int unit = cta; unit < p.n_units; unit += n_cta) {
        wait_full(&tmem_empty_bar[buf], acc_phase ^ 1);           // the epilogue has drained this accumulator pair
        ptx::tc_fence_after();
        uint32_t accumulate = 0;
        const int tile = LINEAR ? unit / p.n_halves : unit;
        const int tidx = p.t0 + (tile / tiles_per_img) % p.T;
        const int rem_m = tile % tiles_per_img;
        const int oy_m = (rem_m / p.tiles_x) * tile_h, ox_m = (rem_m % p.tiles_x) * kTileW;
        for (int grp = 0; grp < n_groups; ++grp) {
          if (!LINEAR && p.skip_t && group_is_padding(p, grp, tidx, oy_m, ox_m, tile_h)) continue;
          const int tap0 = p.gstart[grp], gsz = p.gsize[grp];
          for (int kb = 0; kb < p.kblocks; ++kb) {
            const int k_begin = kb == 0 ? p.ks_first : 0, k_end = kb == p.kblocks - 1 ? p.ks_end : kBK / 16;
            uint32_t a_hi0 = 0;
            if constexpr (!LINEAR) {                     // one activation stage serves the whole group
              wait_full(&a_full[as], aph);
              ptx::tc_fence_after();
              a_hi0 = ptx::smem_u32(a_ring + (size_t)as * a_stage_bytes);
            }
            for (int j = 0; j < gsz; ++j) {
              if constexpr (LINEAR) {                    // one activation stage per tap
                wait_full(&a_full[as], aph);
                ptx::tc_fence_after();
                a_hi0 = ptx::smem_u32(a_ring + (size_t)as * a_stage_bytes);
              }
              const int it = (tap0 + j) * p.kblocks + kb;
              uint32_t b_hi;
              if (resident) {
                b_hi = ptx::smem_u32(b_ring + (size_t)it * p.b_tile_bytes);
              } else {
                wait_full(&b_full[bs], bph);
                ptx::tc_fence_after();
                b_hi = ptx::smem_u32(b_ring + (size_t)bs * p.b_tile_bytes);
              }
              // stacked: db_hi = [W_hi; W_lo] (2*BN rows over the CTA / the pair), db_lo = W_hi alone
              const uint64_t db_hi = ptx::umma_desc_k_sw128(b_hi);
              const uint64_t db_lo = ptx::umma_desc_k_sw128(b_hi + (STACK ? (PAIR ? 2 * kBRows * kBK * 2 : 0) : kBRows * kBK * 2));
              if (ptx::elect_one_sync()) {
              for (int sub = 0; sub < (PAIR ? 1 : p.n_sub); ++sub) {
                // sub-tile rows [sub*8, sub*8+8) of the tile, shifted by j image rows inside the loaded box
                const uint32_t a_hi = a_hi0 + (uint32_t)(((LINEAR ? 0 : j * kTileW) + sub * 128) * 128);
                const uint64_t da_hi = ptx::umma_desc_k_sw128(a_hi), da_lo = ptx::umma_desc_k_sw128(a_hi + p.a_plane_bytes);
                const uint32_t tmem_d = tmem_base + (uint32_t)((buf * 2 + sub) * S::kAccCols);
#pragma unroll
                for (int k = 0; k < kBK / 16; ++k) {
                  if (k < k_begin || k >= k_end) continue;                 // K steps of pure channel padding
                  const uint64_t koff = (uint64_t)((k * 16 * 2) >> 4);     // advance 16 bf16 = 32 bytes along K
                  const uint32_t acc0 = accumulate | (uint32_t)(k > k_begin);
                  if constexpr (STACK) {
                    mma(tmem_d, da_hi + koff, db_hi + koff, idesc2, acc0);                       // A_hi x [W_hi; W_lo]
                    mma(tmem_d, da_lo + koff, db_lo + koff, idesc, 1);                          // A_lo x W_hi
                  } else {
                    mma(tmem_d, da_hi + koff, db_hi + koff, idesc, acc0);
                    mma(tmem_d, da_hi + koff, db_lo + koff, idesc, 1);
                    mma(tmem_d, da_lo + koff, db_hi + koff, idesc, 1);
                  }
                }
              }
              if (!resident) commit(&b_empty[bs]);                // frees the weight slot when these MMAs have read it
              }
              __syncwarp();
              accumulate = 1;
              if (!resident) { if (++bs == p.nb_stages) { bs = 0; bph ^= 1; } }
              if constexpr (LINEAR) {
                if (ptx::elect_one_sync()) commit(&a_empty[as]);                // frees the activation slot
                __syncwarp();
                if (++as == p.na_stages) { as = 0; aph ^= 1; }
              }
            }
            if constexpr (!LINEAR) {
              if (ptx::elect_one_sync()) commit(&a_empty[as]);                  // frees the activation slot
              __syncwarp();
              if (++as == p.na_stages) { as = 0; aph ^= 1; }
            }
          }
        }
        if (ptx::elect_one_sync()) commit(&tmem_full_bar[buf]);                 // accumulators complete -> epilogue
        __syncwarp();
        if (++buf == 2) { buf = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 2) {
    // ===================== epilogue: TMEM -> registers -> global =====================
    const int e = warp - 2;
    const int q = warp & 3;                      // TMEM lane quarter this warp may access (warp id % 4)
    const int half = e >> 2;                     // which half of the BN columns this warp handles
    constexpr int kColsPerWarp = BN / 2;
    const int col0 = half * kColsPerWarp;
    const int r = q * 32 + lane;                 // row of the sub-tile = output pixel
    // destination of this warp's columns (the upper column half may belong to a second tensor)
    const bool second = BN == 128 && half == 1 && p.out2_hi != nullptr;
    __nv_bfloat16* const d_hi = second ? p.out2_hi : p.out_hi;
    __nv_bfloat16* const d_lo = second ? p.out2_lo : p.out_lo;
    const int d_cstride = second ? p.out2_cstride : p.out_cstride;
    const int d_coff = second ? p.out2_coff - 64 : p.out_coff;          // d_coff + column = channel in the destination
    const int d_nstore = second ? 64 + p.n_store2 : p.n_store;
    const bool d_relu = (second ? p.relu2 : p.relu) != 0;
    const bool d_vec = ((p.vec256 >> (second ? 2 : 0)) & 1) != 0;
    int buf = 0; uint32_t acc_phase = 0;
    constexpr bool kSums = BN == 64;              // column sums need kColsPerWarp (= 32) accumulators per thread
    float sacc[kSums ? 32 : 1];
#pragma unroll
    for (int i = 0; i < (kSums ? 32 : 1); ++i) sacc[i] = 0.f;
    int sum_img = -1;
    auto flush_sums = [&](int img_) {             // 32 lanes x 32 columns -> lane l holds column col0 + l (halving butterfly)
      if constexpr (kSums) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
          const bool upper = (lane & off) != 0;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            if (i < off) {
              const float send = upper ? sacc[i] : sacc[i + off];
              const float keep = upper ? sacc[i + off] : sacc[i];
              sacc[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
            }
          }
        }
        p.sum_part[(((size_t)blockIdx.x * 4 + q) * p.n_img + img_) * BN + col0 + lane] = sacc[0];
#pragma unroll
        for (int i = 0; i < 32; ++i) sacc[i] = 0.f;
      }
    };
    ptx::griddep_wait();                          // residual / per-image bias reads and every global write come after
    for (int unit = cta; unit < p.n_units; unit += n_cta) {
      const int tile = LINEAR ? unit / p.n_halves : unit;
      const int ucoff = LINEAR ? (unit % p.n_halves) * BN : 0;   // first column of this unit's half of the convolution
      const int u_coff = d_coff + ucoff, u_nstore = d_nstore - ucoff;
      // 2-D: image of the tile, first image row of this CTA's part and this lane's column; linear: this lane's pixel
      // (img >= n_img past the last pixel)
      int img, oy_t, ox;
      if constexpr (LINEAR) {
        const int m = tile * kLinTile + (int)rank * 128 + r;
        img = m / hw_out;
        const int rem = m - img * hw_out;
        oy_t = rem / p.Wo; ox = rem - oy_t * p.Wo;
      } else {
        img = tile / tiles_per_img;
        const int rem = tile % tiles_per_img;
        oy_t = (rem / p.tiles_x) * tile_h + (int)rank * kSubH; ox = (rem % p.tiles_x) * kTileW + (r & 15);
      }
      auto row_of = [&](int sub) { return LINEAR ? oy_t : oy_t + sub * kSubH + (r >> 4); };
      auto stored = [&](int oy) { return LINEAR ? img < p.n_img : oy < p.Ho && ox < p.Wo; };
      if (kSums && p.sum_part && img != sum_img) {      // tiles come in image order: hand the finished image over
        if (sum_img >= 0) flush_sums(sum_img);
        sum_img = img;
      }
      // latency hiding: the residual of the first chunk and this warp's slice of the per-image bias are requested
      // before waiting for the accumulator; every later residual chunk is requested one chunk ahead
      const int n_sub_eff = PAIR ? 1 : p.n_sub;
      uint32_t nh[8], nl[8];
      auto request_residual = [&](int sub, int j) {
        const int oy = row_of(sub);
        if (stored(oy)) {
          const size_t off = (((size_t)img * p.Ho + oy) * p.Wo + ox) * p.res_cstride + p.res_coff + ucoff + col0 + j * 16;
          // coherent loads: the residual (like the per-image bias below) is written by a PRECEDING kernel that this grid
          // may overlap under programmatic dependent launch, so the read-only (.nc) path is not allowed for it
          if (p.vec256 & 2) {
            ptx::ld_global_v8(p.res_hi + off, nh);
            ptx::ld_global_v8(p.res_lo + off, nl);
          } else {
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              const uint4 h4 = ptx::ld_global_v4(reinterpret_cast<const uint4*>(p.res_hi + off) + g);
              const uint4 l4 = ptx::ld_global_v4(reinterpret_cast<const uint4*>(p.res_lo + off) + g);
              nh[4 * g] = h4.x; nh[4 * g + 1] = h4.y; nh[4 * g + 2] = h4.z; nh[4 * g + 3] = h4.w;
              nl[4 * g] = l4.x; nl[4 * g + 1] = l4.y; nl[4 * g + 2] = l4.z; nl[4 * g + 3] = l4.w;
            }
          }
        }
      };
      if (p.res_mode) request_residual(0, 0);
      const float* bsrc = s_bias + ucoff;         // bias of column c at bsrc[c]
      if (p.img_bias) {
        const float* ib = p.img_bias + (size_t)img * p.img_bias_stride + col0;
        float* wb = s_wb + e * 64;
        __syncwarp();                             // every lane is done with the previous tile's slice
#pragma unroll
        for (int i = lane; i < kColsPerWarp; i += 32) wb[i] = *(reinterpret_cast<const volatile float*>(ib) + i);
        __syncwarp();
        bsrc = wb - col0;
      }
      ptx::mbar_wait(&tmem_full_bar[buf], acc_phase);
      ptx::tc_fence_after();
#pragma unroll 1
      for (int sub = 0; sub < n_sub_eff; ++sub) {
        const int oy = row_of(sub);
        const bool valid = stored(oy);
        const size_t pix = ((size_t)img * p.Ho + oy) * p.Wo + ox;
        float hacc[kMaxHeadOut];
#pragma unroll
        for (int k = 0; k < kMaxHeadOut; ++k) hacc[k] = 0.f;
        const uint32_t tmem_acc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((buf * 2 + sub) * S::kAccCols + col0);
#pragma unroll 1
        for (int j = 0; j < kColsPerWarp / 16; ++j) {
          const int cb = col0 + j * 16;              // first output channel of this chunk
          uint32_t acc[16];
          uint32_t acc2[16];                         // stacked operand: the hi x lo products live n_mma columns further
          const bool computed = cb < p.n_mma;        // columns beyond n_mma: zero weights, never multiplied
          if (computed) {
            ptx::tmem_ld_32x32b_x16(tmem_acc + j * 16, acc);
            if constexpr (STACK) ptx::tmem_ld_32x32b_x16(tmem_acc + p.n_mma + j * 16, acc2);
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) { acc[i] = 0u; acc2[i] = 0u; }
          }
          uint32_t rhw[8], rlw[8];                   // residual of this chunk (requested one chunk ago)
          if (p.res_mode) {
#pragma unroll
            for (int i = 0; i < 8; ++i) { rhw[i] = nh[i]; rlw[i] = nl[i]; }
            const bool last_j = j + 1 == kColsPerWarp / 16;
            if (!last_j) request_residual(sub, j + 1);
            else if (sub + 1 < n_sub_eff) request_residual(sub + 1, 0);
          }
          ptx::tmem_ld_wait();
          if (valid) {
            float v[16];
#pragma unroll
            for (int g = 0; g < 4; ++g) {          // bias: per-image slice (conv bias already folded in) or the conv's own
              const float4 b4 = *reinterpret_cast<const float4*>(bsrc + cb + 4 * g);
              if constexpr (STACK) {
                v[4 * g + 0] = (__uint_as_float(acc[4 * g + 0]) + __uint_as_float(acc2[4 * g + 0])) + b4.x;
                v[4 * g + 1] = (__uint_as_float(acc[4 * g + 1]) + __uint_as_float(acc2[4 * g + 1])) + b4.y;
                v[4 * g + 2] = (__uint_as_float(acc[4 * g + 2]) + __uint_as_float(acc2[4 * g + 2])) + b4.z;
                v[4 * g + 3] = (__uint_as_float(acc[4 * g + 3]) + __uint_as_float(acc2[4 * g + 3])) + b4.w;
              } else {
                v[4 * g + 0] = __uint_as_float(acc[4 * g + 0]) + b4.x;
                v[4 * g + 1] = __uint_as_float(acc[4 * g + 1]) + b4.y;
                v[4 * g + 2] = __uint_as_float(acc[4 * g + 2]) + b4.z;
                v[4 * g + 3] = __uint_as_float(acc[4 * g + 3]) + b4.w;
              }
            }
            if (p.res_mode) {
#pragma unroll
              for (int e2 = 0; e2 < 8; ++e2) {
                const float r0 = __uint_as_float(rhw[e2] << 16) + __uint_as_float(rlw[e2] << 16);
                const float r1 = __uint_as_float(rhw[e2] & 0xFFFF0000u) + __uint_as_float(rlw[e2] & 0xFFFF0000u);
                float& a0 = v[e2 * 2], &a1 = v[e2 * 2 + 1];
                if (p.res_mode == 1) { a0 += r0; a1 += r1; if (d_relu) { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); } }
                else { if (d_relu) { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); } a0 += r0; a1 += r1; }
              }
            } else if (d_relu) {
#pragma unroll
              for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
            }
            if (d_hi && cb < u_nstore) {
              __nv_bfloat16* ohp = d_hi + pix * d_cstride + u_coff + cb;
              __nv_bfloat16* olp = d_lo + pix * d_cstride + u_coff + cb;
              uint32_t hw[8], lw[8];
#pragma unroll
              for (int e2 = 0; e2 < 8; ++e2) {
                const float x0 = v[e2 * 2], x1 = v[e2 * 2 + 1];
                const uint32_t h = ptx::pack_bf16x2(x0, x1);                   // one cvt.rn.bf16x2.f32
                const float r0 = x0 - __uint_as_float(h << 16), r1 = x1 - __uint_as_float(h & 0xFFFF0000u);
                hw[e2] = h;
                lw[e2] = ptx::pack_bf16x2(r0, r1);
              }
              if (d_vec && cb + 16 <= u_nstore) {               // one full 32-byte sector per plane and lane
                ptx::st_global_v8(ohp, hw);
                ptx::st_global_v8(olp, lw);
              } else {
                reinterpret_cast<uint4*>(ohp)[0] = make_uint4(hw[0], hw[1], hw[2], hw[3]);
                reinterpret_cast<uint4*>(olp)[0] = make_uint4(lw[0], lw[1], lw[2], lw[3]);
                if (cb + 8 < u_nstore) {
                  reinterpret_cast<uint4*>(ohp)[1] = make_uint4(hw[4], hw[5], hw[6], hw[7]);
                  reinterpret_cast<uint4*>(olp)[1] = make_uint4(lw[4], lw[5], lw[6], lw[7]);
                }
              }
            }
            if (p.out_f32 && p.f32_nhwc) {
              const int c0 = p.f32_coff + ucoff + cb;
              float* dst = p.out_f32 + pix * p.n_valid + c0;
              if (c0 + 16 <= p.n_valid && (p.n_valid & 7) == 0) {          // rows are 32-byte aligned (host checks the base)
                ptx::st_global_v8f(dst, v);
                ptx::st_global_v8f(dst + 8, v + 8);
              } else {
#pragma unroll
                for (int i = 0; i < 16; ++i)
                  if (c0 + i < p.n_valid) dst[i] = v[i];
              }
            } else if (p.out_f32) {
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const int c = p.f32_coff + ucoff + cb + i;
                if (c < p.n_valid) {
                  float x = v[i];
                  if (p.sigmoid) x = 1.f / (1.f + __expf(-x));
                  p.out_f32[(((size_t)img * p.n_valid + c) * p.Ho + oy) * p.Wo + ox] = x;
                }
              }
            }
            if constexpr (kSums) {
              if (p.sum_part) {
                if (j == 0) {
#pragma unroll
                  for (int i = 0; i < 16; ++i) sacc[i] += v[i];
                } else {
#pragma unroll
                  for (int i = 0; i < 16; ++i) sacc[16 + i] += v[i];
                }
              }
            }
            if (p.head_ko) {
#pragma unroll
              for (int k = 0; k < kMaxHeadOut; ++k) {
                if (k < p.head_ko) {
                  const float* w = s_head + k * BN + cb;
                  float a = hacc[k];
#pragma unroll
                  for (int i = 0; i < 16; ++i) a = fmaf(w[i], v[i], a);
                  hacc[k] = a;
                }
              }
            }
          }
        }
        if (p.head_ko) {
          // the two column halves of a pixel live in two warps of the same lane quarter: the upper half hands its
          // partial dot products over through shared memory (named barrier of the 64 threads involved)
          if (half == 1) {
#pragma unroll
            for (int k = 0; k < kMaxHeadOut; ++k) if (k < p.head_ko) s_hx[k * 128 + r] = hacc[k];
          }
          asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
          if (half == 0 && valid) {
#pragma unroll
            for (int k = 0; k < kMaxHeadOut; ++k) {
              if (k < p.head_ko) {
                float x = hacc[k] + s_hx[k * 128 + r] + p.head_b[k];
                if (p.head_sigmoid_mask & (1 << k)) x = 1.f / (1.f + __expf(-x));
                p.head_out[k][(size_t)img * p.head_img_stride[k] + (size_t)oy * p.Wo + ox] = x;
              }
            }
          }
          asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
        }
      }
      // this warp has finished reading the accumulator pair
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (PAIR) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&tmem_empty_bar[buf]), 0));
        else ptx::mbar_arrive(&tmem_empty_bar[buf]);
      }
      if (++buf == 2) { buf = 0; acc_phase ^= 1; }
    }
    if (kSums && p.sum_part && sum_img >= 0) flush_sums(sum_img);
  }
  ptx::tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) ptx::cluster_sync();        // the peer may still be reading this CTA's operands / signalling its barriers
  if (warp == 1) {
    if constexpr (PAIR) ptx::tmem_dealloc_pair<S::kTmemCols>(tmem_base);
    else ptx::tmem_dealloc<S::kTmemCols>(tmem_base);
  }
}

// col_sums[img][c] = sum over the (CTA, lane quarter) partial rows, in a fixed order: block (bn, 16) -- 16 slices of the
// partial rows, independent loads issued in batches, then a fixed-order sum of the slices through shared memory
__global__ void col_sum_reduce_kernel(const float* __restrict__ part, int n_part, int n_img, int bn,
                                      float* __restrict__ out) {
  __shared__ float sm[16][64];
  ptx::griddep_launch_dependents();
  ptx::griddep_wait();                      // the partial rows come from the convolution just before
  const int img = blockIdx.x, c = threadIdx.x, sl = threadIdx.y;
  const int per = (n_part + 15) / 16;
  const int k0 = sl * per, k1 = min(n_part, k0 + per);
  float a = 0.f;
  for (int kb = k0; kb < k1; kb += 8) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = kb + i < k1 ? part[((size_t)(kb + i) * n_img + img) * bn + c] : 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) a += v[i];
  }
  sm[sl][c] = a;
  __syncthreads();
  if (sl == 0) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) t += sm[i][c];
    out[(size_t)img * bn + c] = t;
  }
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_tmapEncodeTiled encode_fn() {
  static PFN_tmapEncodeTiled fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tmapEncodeTiled>(ptr);
  }
  return fn;
}

typedef CUresult (*PFN_tmapEncodeIm2col)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                         const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                         const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                         CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_tmapEncodeIm2col encode_im2col_fn() {
  static PFN_tmapEncodeIm2col fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tmapEncodeIm2col>(ptr);
  }
  return fn;
}

int launch_col_sum_reduce(const float* part, int n_part, int n_img, float* out, cudaStream_t stream) {
  STP3_CUDA_OK(launch_pdl(col_sum_reduce_kernel, dim3(n_img), dim3(64, 16), 0, stream, part, n_part, n_img, 64, out));
  return STP3_OK;
}

}  // namespace stp3

using namespace stp3;

static int conv_num_sms() {
  static const int n = [] {
    int dev = 0, v = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v;
  }();
  return n;
}

extern "C" size_t stp3_conv_col_sums_scratch_bytes(int n_img, int bn) {
  return (size_t)conv_num_sms() * 4 * (size_t)(n_img > 0 ? n_img : 0) * (size_t)(bn > 0 ? bn : 0) * sizeof(float);
}

extern "C" int stp3_conv_fwd(const stp3_conv_desc* d, const void* x_hi, const void* x_lo, const void* w,
                             const float* bias, const float* img_bias, const void* res_hi, const void* res_lo,
                             void* y_hi, void* y_lo, float* y_f32, const stp3_conv_head* head, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  STP3_CHECK_ARG(d && x_hi && x_lo && w && bias, "stp3_conv_fwd: null pointer argument");
  STP3_CHECK_ARG((y_hi && y_lo) || y_f32 || head, "stp3_conv_fwd: no output tensor");
  if (head) {
    STP3_CHECK_ARG(head->n_out >= 1 && head->n_out <= kMaxHeadOut && head->w && head->b, "bad fused head");
    STP3_CHECK_ARG(d->bn <= 128, "a fused head needs bn <= 128");
    for (int k = 0; k < head->n_out; ++k) STP3_CHECK_ARG(head->out[k] != nullptr, "fused head: null output plane");
  }
  STP3_CHECK_ARG(d->B > 0 && d->T > 0 && d->H > 0 && d->W > 0 && d->Ho > 0 && d->Wo > 0, "non-positive dimension");
  const int T_total = d->T_total > 0 ? d->T_total : d->T;
  STP3_CHECK_ARG(d->t0 >= 0 && d->t0 + d->T <= T_total, "frame window [t0, t0+T) outside the input tensor");
  const int n_store = d->n_store > 0 ? d->n_store : d->bn;
  STP3_CHECK_ARG(n_store % 8 == 0 && n_store <= d->bn, "n_store must be a multiple of 8 and <= bn");
  STP3_CHECK_ARG(d->in_cstride % 64 == 0 && d->cin % 64 == 0 && d->cin_off % 64 == 0 && d->cin > 0 &&
                 d->cin_off + d->cin <= d->in_cstride, "input channels must be padded to multiples of 64");
  STP3_CHECK_ARG(d->bn == 64 || d->bn == 128 || d->bn == 256, "bn (padded output channels) must be 64, 128 or 256");
  STP3_CHECK_ARG(d->stride == 1 || d->stride == 2, "stride must be 1 or 2");
  STP3_CHECK_ARG(d->ntaps >= 1 && d->ntaps <= kMaxTaps, "ntaps out of range");
  if (y_hi) STP3_CHECK_ARG(d->out_cstride % 8 == 0 && d->out_coff % 8 == 0 && d->out_coff + n_store <= d->out_cstride,
                           "output channel window does not fit the output tensor");
  if (d->res_mode) STP3_CHECK_ARG(res_hi && res_lo && d->res_cstride % 8 == 0 && d->res_coff % 8 == 0 &&
                                  d->res_coff + d->bn <= d->res_cstride, "bad residual tensor");
  if (y_f32) STP3_CHECK_ARG(d->n_valid > 0 && d->n_valid <= d->bn, "n_valid out of range");
  PFN_tmapEncodeTiled enc = encode_fn();
  if (!enc) return set_error(STP3_ECUDA, "cuTensorMapEncodeTiled is not available from the driver");

  // tuning knobs (0 = automatic): desc->tune_n_sub / tune_group, or the STP3_CONV_NSUB / STP3_CONV_GROUP environment
  static const int env_nsub = [] { const char* e = getenv("STP3_CONV_NSUB"); return e ? atoi(e) : 0; }();
  static const int env_group = [] { const char* e = getenv("STP3_CONV_GROUP"); return e ? atoi(e) : 0; }();
  const int want_nsub = d->tune_n_sub ? d->tune_n_sub : env_nsub;
  const int want_group_raw = d->tune_group ? d->tune_group : env_group;
  const int want_group = want_group_raw & 3;
  static const bool use_pdl = stp3_pdl_enabled("STP3_CONV_PDL");
  const bool stream_weights = (want_group_raw & 4) != 0;    // +4: keep the weights in the ring even if they would fit
  // +8: stacked [W_hi; W_lo] operand (bn = 64 only).  Untuned (tune_group == 0) multi-tap 64-column layers use it: it
  // won on every such layer of the hot path (profiles/r01_autotune_v9.txt)
  const bool stack = d->bn == 64 && ((want_group_raw & 8) != 0 || (want_group_raw == 0 && d->ntaps > 1));
  // taps that can share one activation load: runs (<= 4) of consecutive taps with the same (dt, dx) and dy advancing
  // by the stride
  ConvParams p;
  p.n_groups = 0; p.gmax = 1;
  for (int i = 0; i < d->ntaps;) {
    int g = 1;
    if (want_group != 1)
      while (g < 4 && i + g < d->ntaps && d->taps[i + g][0] == d->taps[i][0] && d->taps[i + g][2] == d->taps[i][2] &&
             d->taps[i + g][1] == d->taps[i][1] + g * d->stride)
        ++g;
    p.gstart[p.n_groups] = (unsigned char)i; p.gsize[p.n_groups] = (unsigned char)g; ++p.n_groups;
    if (g > p.gmax) p.gmax = g;
    i += g;
  }
  const int group = p.gmax;
  // two sub-tiles per tile halve the weight traffic; small images keep one so that there are enough tiles
  const int n_img_ = d->B * d->T;
  const long long tiles16 = (long long)n_img_ * ceil_div(d->Wo, kTileW) * ceil_div(d->Ho, 2 * kSubH);
  // tune_n_sub == 3: the 16x16 tile is shared by a CTA pair (cta_group::2), 8 image rows per CTA
  // untuned (tune_n_sub == 0) multi-tap layers take the pair tiling, the autotuner's choice on all of them
  // tune_n_sub == 4 / 5: linear tiling, 128 consecutive output pixels per CTA / 256 per CTA pair (see the kernel)
  const bool linear = want_nsub == 4 || want_nsub == 5;
  const bool pair = want_nsub == 3 || want_nsub == 5 || (want_nsub == 0 && d->ntaps > 1);
  const int n_sub = pair || linear ? 1 : (want_nsub == 1 || want_nsub == 2 ? want_nsub : (tiles16 >= 3 * 148 ? 2 : 1));
  const int tile_h = pair ? 2 * kSubH : kSubH * n_sub;
  const int box_h = kSubH * n_sub + (group - 1);                         // image rows one CTA loads per stage

  CUtensorMap tm_hi, tm_lo, tm_w;
  int lin_lo_w = 0, lin_lo_h = 0;
  if (linear) {
    STP3_CHECK_ARG(d->t0 == 0 && d->T == T_total, "linear tiling: every frame of the input tensor (no frame window)");
    STP3_CHECK_ARG(!d->col_sums && !head && !img_bias && !y_f32,
                   "linear tiling: no col_sums, fused head, per-image bias or fp32 output");
    int hi_w = d->taps[0][2], hi_h = d->taps[0][1];
    lin_lo_w = hi_w; lin_lo_h = hi_h;
    for (int i = 0; i < d->ntaps; ++i) {
      STP3_CHECK_ARG(d->taps[i][0] == 0, "linear tiling: 2-D taps only (dt = 0)");
      lin_lo_w = d->taps[i][2] < lin_lo_w ? d->taps[i][2] : lin_lo_w; hi_w = d->taps[i][2] > hi_w ? d->taps[i][2] : hi_w;
      lin_lo_h = d->taps[i][1] < lin_lo_h ? d->taps[i][1] : lin_lo_h; hi_h = d->taps[i][1] > hi_h ? d->taps[i][1] : hi_h;
    }
    // bounding box of the traversal: the first input pixel of every output pixel's window (tap at the lower corner),
    // [lo, dim - 1 + up] walked with the conv stride, so that it holds exactly Wo x Ho start pixels
    const int up_w = (d->Wo - 1) * d->stride + lin_lo_w - (d->W - 1);
    const int up_h = (d->Ho - 1) * d->stride + lin_lo_h - (d->H - 1);
    auto in8 = [](int v) { return v >= -128 && v <= 127; };
    STP3_CHECK_ARG(in8(lin_lo_w) && in8(lin_lo_h) && in8(up_w) && in8(up_h) && hi_w - lin_lo_w < 256 &&
                   hi_h - lin_lo_h < 256, "linear tiling: padding / output size outside the im2col corner range [-128, 127]");
    PFN_tmapEncodeIm2col enc2 = encode_im2col_fn();
    if (!enc2) return set_error(STP3_ECUDA, "cuTensorMapEncodeIm2col is not available from the driver");
    const cuuint64_t dims[4] = {(cuuint64_t)d->in_cstride, (cuuint64_t)d->W, (cuuint64_t)d->H,
                                (cuuint64_t)d->B * T_total};
    const cuuint64_t strides[3] = {(cuuint64_t)d->in_cstride * 2, (cuuint64_t)d->W * d->in_cstride * 2,
                                   (cuuint64_t)d->H * d->W * d->in_cstride * 2};
    const int lower[2] = {lin_lo_w, lin_lo_h}, upper[2] = {up_w, up_h};          // innermost (W) first
    const cuuint32_t estr[4] = {1, (cuuint32_t)d->stride, (cuuint32_t)d->stride, 1};
    CUresult r1 = enc2(&tm_hi, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x_hi), dims, strides, lower, upper,
                       kBK, 128, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CUresult r2 = enc2(&tm_lo, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x_lo), dims, strides, lower, upper,
                       kBK, 128, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r1 != CUDA_SUCCESS || r2 != CUDA_SUCCESS)
      return set_error(STP3_ECUDA, "cuTensorMapEncodeIm2col(activation) failed: %d %d", (int)r1, (int)r2);
  } else {
    const cuuint64_t dims[5] = {(cuuint64_t)d->in_cstride, (cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)T_total,
                                (cuuint64_t)d->B};
    const cuuint64_t strides[4] = {(cuuint64_t)d->in_cstride * 2, (cuuint64_t)d->W * d->in_cstride * 2,
                                   (cuuint64_t)d->H * d->W * d->in_cstride * 2,
                                   (cuuint64_t)T_total * d->H * d->W * d->in_cstride * 2};
    const cuuint32_t box[5] = {(cuuint32_t)kBK, (cuuint32_t)((kTileW - 1) * d->stride + 1),
                               (cuuint32_t)((box_h - 1) * d->stride + 1), 1, 1};
    const cuuint32_t estr[5] = {1, (cuuint32_t)d->stride, (cuuint32_t)d->stride, 1, 1};
    CUresult r1 = enc(&tm_hi, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(x_hi), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CUresult r2 = enc(&tm_lo, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(x_lo), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r1 != CUDA_SUCCESS || r2 != CUDA_SUCCESS)
      return set_error(STP3_ECUDA, "cuTensorMapEncodeTiled(activation) failed: %d %d", (int)r1, (int)r2);
  }
  const int kblocks = d->cin / kBK;
  const int bn_launch = d->bn == 256 ? 128 : d->bn;     // 256 output channels: two 128-column launches (2-D tiling)
  const int n_halves = linear && d->bn == 256 ? 2 : 1;  // or one linear launch whose work units cover both halves
  // the MMAs cover only the columns that carry weights (n_cols, rounded up to the UMMA granularity of 16)
  const int n_mma = d->bn <= 128 && d->n_cols > 0 && d->n_cols < d->bn ? ((d->n_cols + 15) / 16) * 16 : bn_launch;
  {
    const cuuint64_t dims[2] = {(cuuint64_t)kBK, (cuuint64_t)d->ntaps * kblocks * 2 * d->bn};
    const cuuint64_t strides[1] = {(cuuint64_t)kBK * 2};
    const cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)(pair ? n_mma / 2 : n_mma)};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&tm_w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(w), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(STP3_ECUDA, "cuTensorMapEncodeTiled(weights) failed: %d", (int)r);
  }

  p.n_img = d->B * d->T; p.T = d->T; p.t0 = d->t0; p.Ho = d->Ho; p.Wo = d->Wo;
  p.T_total = T_total;
  p.H = d->H; p.W = d->W;
  p.skip_t = 0;                                     // safe only if some tap always stays inside: the centre tap
  for (int i = 0; i < d->ntaps; ++i) if (d->taps[i][0] == 0 && d->taps[i][1] == 0 && d->taps[i][2] == 0) p.skip_t = 1;
  p.m_total = 0; p.lin_lo_w = lin_lo_w; p.lin_lo_h = lin_lo_h; p.n_halves = n_halves;
  p.tiles_x = ceil_div(d->Wo, kTileW); p.tiles_y = ceil_div(d->Ho, tile_h); p.n_sub = n_sub;
  p.stride = d->stride; p.kblocks = kblocks; p.cin_off = d->cin_off; p.ntaps = d->ntaps;
  {
    const int k_lo = d->k_hi > 0 ? d->k_lo : 0, k_hi = d->k_hi > 0 ? d->k_hi : d->cin;
    STP3_CHECK_ARG(k_lo % 16 == 0 && k_hi % 16 == 0 && k_lo >= 0 && k_lo < k_hi && k_hi <= d->cin &&
                   k_lo < kBK && k_hi > d->cin - kBK, "k_lo / k_hi: multiples of 16 inside the first / last 64-channel block");
    p.ks_first = k_lo / 16;
    p.ks_end = (k_hi - (kblocks - 1) * kBK) / 16;
    STP3_CHECK_ARG(kblocks > 1 || p.ks_first < p.ks_end, "empty K range");
  }
  p.a_plane_bytes = (linear ? 128 : box_h * kTileW) * kBK * 2; p.w_rows = d->bn; p.n_mma = n_mma;
  for (int i = 0; i < d->ntaps; ++i) { p.tap[i][0] = d->taps[i][0]; p.tap[i][1] = d->taps[i][1]; p.tap[i][2] = d->taps[i][2]; p.tap[i][3] = 0; }
  p.relu = d->relu; p.res_mode = d->res_mode;
  p.res_hi = static_cast<const __nv_bfloat16*>(res_hi); p.res_lo = static_cast<const __nv_bfloat16*>(res_lo);
  p.res_cstride = d->res_cstride;
  p.out_hi = static_cast<__nv_bfloat16*>(y_hi); p.out_lo = static_cast<__nv_bfloat16*>(y_lo);
  p.out_cstride = d->out_cstride;
  p.out2_hi = static_cast<__nv_bfloat16*>(d->y2_hi); p.out2_lo = static_cast<__nv_bfloat16*>(d->y2_lo);
  p.out2_cstride = d->out2_cstride; p.out2_coff = d->out2_coff; p.relu2 = d->relu2;
  p.n_store2 = d->n_store2 > 0 ? d->n_store2 : 64;
  if (d->y2_hi) {
    STP3_CHECK_ARG(d->bn == 128 && d->y2_lo && y_hi && !d->res_mode && !head && !y_f32 && !d->col_sums,
                   "second destination: 128-column convolutions with plain hi/lo outputs only");
    STP3_CHECK_ARG(n_store <= 64 && p.n_store2 % 8 == 0 && p.n_store2 <= 64 && d->out2_cstride % 8 == 0 &&
                   d->out2_coff % 8 == 0 && d->out2_coff + p.n_store2 <= d->out2_cstride,
                   "second destination: channel window does not fit");
  }
  p.out_f32 = y_f32; p.n_valid = d->n_valid; p.sigmoid = d->sigmoid;
  p.f32_nhwc = d->f32_layout;
  STP3_CHECK_ARG(d->f32_layout == 0 || d->f32_layout == 1, "f32_layout must be 0 (n_img, n_valid, Ho, Wo) or 1 (n_img, Ho, Wo, n_valid)");
  if (y_f32 && d->f32_layout == 1)
    STP3_CHECK_ARG((reinterpret_cast<uintptr_t>(y_f32) & 31) == 0 && !d->sigmoid,
                   "channels-last y_f32 must be 32-byte aligned (and carries no sigmoid)");
  p.img_bias_stride = d->bn;
  p.head_ko = 0; p.head_w = nullptr; p.head_b = nullptr; p.head_sigmoid_mask = 0;
  for (int k = 0; k < kMaxHeadOut; ++k) { p.head_out[k] = nullptr; p.head_img_stride[k] = 0; }
  if (head) {
    p.head_ko = head->n_out; p.head_w = head->w; p.head_b = head->b; p.head_sigmoid_mask = head->sigmoid_mask;
    for (int k = 0; k < head->n_out; ++k) { p.head_out[k] = head->out[k]; p.head_img_stride[k] = head->img_stride[k]; }
  }
  const int k_iters = d->ntaps * kblocks;
  const long long m_total = (long long)p.n_img * d->Ho * d->Wo;
  const long long n_tiles = linear ? (m_total + (pair ? 255 : 127)) / (pair ? 256 : 128) : (long long)p.n_img * p.tiles_x * p.tiles_y;
  const long long nblk = n_tiles * n_halves;                                    // work units
  STP3_CHECK_ARG(nblk > 0 && m_total < (1ll << 31) && nblk < (1ll << 31), "grid too large");
  p.n_tiles = (int)n_tiles; p.n_units = (int)nblk; p.m_total = (int)m_total;
  const int num_sms = conv_num_sms();
  unsigned grid = (unsigned)(nblk < num_sms ? nblk : num_sms);           // persistent: one CTA per SM
  if (pair) grid = 2u * (unsigned)(nblk < num_sms / 2 ? nblk : num_sms / 2);
  const size_t smem_cap = 227 * 1024;
  const size_t a_stage = 2 * (size_t)p.a_plane_bytes;

  int launched_grid = (int)grid;
  p.sum_part = nullptr;
  if (d->col_sums) {
    STP3_CHECK_ARG(d->bn == 64, "col_sums: 64-column convolutions only");
    STP3_CHECK_ARG(d->col_sums_scratch && d->col_sums_scratch_bytes >= stp3_conv_col_sums_scratch_bytes(p.n_img, 64),
                   "col_sums: scratch buffer missing or smaller than stp3_conv_col_sums_scratch_bytes()");
    p.sum_part = static_cast<float*>(d->col_sums_scratch);
    // CTAs that never see an image leave its partial rows untouched: start from zeros
    STP3_CUDA_OK(cudaMemsetAsync(p.sum_part, 0, (size_t)grid * 4 * p.n_img * 64 * sizeof(float), stream));
  }

  for (int part = 0; part * bn_launch * n_halves < d->bn; ++part) {
    const int coff = part * bn_launch;
    p.w_row_off = coff;
    p.bias = bias + coff;
    p.img_bias = img_bias ? img_bias + coff : nullptr;
    p.res_coff = d->res_coff + coff;
    p.out_coff = d->out_coff + coff;
    p.n_store = n_store - coff < bn_launch * n_halves ? (n_store - coff > 0 ? n_store - coff : 0) : bn_launch * n_halves;
    p.f32_coff = coff;
    auto al32 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 31) == 0; };
    p.vec256 = (y_hi && d->out_cstride % 16 == 0 && p.out_coff % 16 == 0 && al32(y_hi) && al32(y_lo) ? 1 : 0) |
               (d->res_mode && d->res_cstride % 16 == 0 && p.res_coff % 16 == 0 && al32(res_hi) && al32(res_lo) ? 2 : 0) |
               (d->y2_hi && d->out2_cstride % 16 == 0 && d->out2_coff % 16 == 0 && al32(d->y2_hi) && al32(d->y2_lo) ? 4 : 0);
#define STP3_LAUNCH_CONV(BN_, PAIR_, STACK_, LIN_)                                                                \
    do {                                                                                                          \
      using SM = ConvSmem<BN_, PAIR_, STACK_, LIN_>;                                                                  \
      p.b_rows = PAIR_ ? n_mma / 2 : n_mma;                                                                       \
      p.b_tile_bytes = (STACK_ && PAIR_ ? 3 : 2) * p.b_rows * kBK * 2;                                            \
      const size_t avail = smem_cap - 1024 - SM::tail_bytes();                                                    \
      const size_t wbytes = (size_t)k_iters * (size_t)p.b_tile_bytes;                                                    \
      /* small weight tensors stay resident in smem next to >= 2 activation stages */                            \
      const bool res = !stream_weights && n_halves == 1 && wbytes + 2 * a_stage <= avail;                                        \
      int na, nb;                                                                                                 \
      if (res) {                                                                                                  \
        na = (int)((avail - wbytes) / a_stage); nb = 0;                                                           \
      } else {                                                                                                    \
        /* as many activation stages as fit beside max(2, group) weight slots, then fill up with weight slots */  \
        const int nb_min = group > 2 ? group : 2;                                                                 \
        na = (int)((avail - (size_t)nb_min * (size_t)p.b_tile_bytes) / a_stage);                                         \
        if (na < 2) na = 2;                                                                                       \
        if (na > kMaxAStages) na = kMaxAStages;                                                                   \
        if ((size_t)na * a_stage + 2 * (size_t)p.b_tile_bytes > avail)                                                   \
          return set_error(STP3_EUNSUPPORTED, "convolution does not fit in shared memory");                       \
        nb = (int)((avail - (size_t)na * a_stage) / (size_t)p.b_tile_bytes);                                             \
      }                                                                                                           \
      if (na > kMaxAStages) na = kMaxAStages;                                                                     \
      if (nb > kMaxBStages) nb = kMaxBStages;                                                                     \
      p.na_stages = na; p.nb_stages = nb; p.b_resident = res ? 1 : 0;                                             \
      const size_t smem_bytes = 1024 + na * a_stage + (res ? wbytes : (size_t)nb * (size_t)p.b_tile_bytes) + SM::tail_bytes(); \
      auto kern = conv_igemm_kernel<BN_, PAIR_, STACK_, LIN_>;                                                        \
      /* once per kernel instantiation and device: the attribute call costs microseconds on every eager launch */ \
      static thread_local int attr_dev = -1;                                                                      \
      int cur_dev = 0; cudaGetDevice(&cur_dev);                                                                   \
      if (attr_dev != cur_dev) {                                                                                  \
        STP3_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap));     \
        attr_dev = cur_dev;                                                                                       \
      }                                                                                                           \
      cudaLaunchConfig_t cfg = {};                                                                                \
      cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kConvThreads);                                                \
      cfg.dynamicSmemBytes = smem_bytes; cfg.stream = stream;                                                     \
      cudaLaunchAttribute attr[2];                                                                                \
      attr[0].id = cudaLaunchAttributeClusterDimension;                                                           \
      attr[0].val.clusterDim.x = PAIR_ ? 2 : 1; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;       \
      cfg.attrs = attr; cfg.numAttrs = PAIR_ ? 1 : 0;                                                             \
      if (PAIR_) {                                                                                                \
        /* co-resident pairs the device can host with this much shared memory (GPCs with an odd SM count) */      \
        /* depends on the kernel and its shared-memory size only: cached per (device, smem size) */               \
        static thread_local int occ_dev = -1, occ_val = 0; static thread_local size_t occ_smem = 0;               \
        int max_clusters = occ_val;                                                                               \
        if (occ_dev != cur_dev || occ_smem != smem_bytes) {                                                       \
          STP3_CUDA_OK(cudaOccupancyMaxActiveClusters(&max_clusters, kern, &cfg));                                \
          occ_dev = cur_dev; occ_smem = smem_bytes; occ_val = max_clusters;                                       \
        }                                                                                                         \
        if (max_clusters < 1) return set_error(STP3_EUNSUPPORTED, "no CTA pair fits on this device");             \
        if (cfg.gridDim.x > 2u * (unsigned)max_clusters) cfg.gridDim.x = 2u * (unsigned)max_clusters;             \
      }                                                                                                           \
      if (use_pdl) {                                                                                              \
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                                          \
        attr[0].val.programmaticStreamSerializationAllowed = 1;                                                   \
        attr[1].id = cudaLaunchAttributeClusterDimension;                                                         \
        attr[1].val.clusterDim.x = PAIR_ ? 2 : 1; attr[1].val.clusterDim.y = 1; attr[1].val.clusterDim.z = 1;     \
        cfg.numAttrs = PAIR_ ? 2 : 1;                                                                             \
      }                                                                                                           \
      launched_grid = (int)cfg.gridDim.x;                                                                         \
      STP3_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, tm_hi, tm_lo, tm_w, p));                                        \
    } while (0)
#define STP3_DISPATCH_CONV(LIN_)                                                                                  \
    if (bn_launch == 64) {                                                                                        \
      if (stack) { if (pair) STP3_LAUNCH_CONV(64, true, true, LIN_); else STP3_LAUNCH_CONV(64, false, true, LIN_); } \
      else { if (pair) STP3_LAUNCH_CONV(64, true, false, LIN_); else STP3_LAUNCH_CONV(64, false, false, LIN_); }  \
    } else {                                                                                                      \
      if (pair) STP3_LAUNCH_CONV(128, true, false, LIN_); else STP3_LAUNCH_CONV(128, false, false, LIN_);         \
    }
    if (linear) { STP3_DISPATCH_CONV(true) } else { STP3_DISPATCH_CONV(false) }
#undef STP3_DISPATCH_CONV
#undef STP3_LAUNCH_CONV
    STP3_CUDA_OK(cudaGetLastError());
  }
  if (p.sum_part) {
    STP3_CUDA_OK(launch_pdl(col_sum_reduce_kernel, dim3(p.n_img), dim3(64, 16), 0, stream, (const float*)p.sum_part,
                            launched_grid * 4, p.n_img, 64, static_cast<float*>(d->col_sums)));
  }
  return STP3_OK;
}
