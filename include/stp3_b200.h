/* stp3_b200 — C ABI of the B200-native (sm_100a) ST-P3 camera->BEV perception hot path.
 *
 * The reference (OpenDriveLab/ST-P3) is 100 % Python/PyTorch and has no FFI of its own; the drop-in boundary is
 * the nn.Module surface (SURVEY.md §8b).  This header is the C boundary that sits directly underneath those
 * modules: each entry point names the reference interface it replaces (file:line under /root/reference).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch's caching allocator in practice), unless the
 *     parameter is documented as a host value;
 *   - no entry point allocates, frees or synchronises: work is enqueued on `stream` (a cudaStream_t passed as
 *     void*) and the call returns immediately;
 *   - return value: 0 on success, a negative STP3_E* code otherwise; stp3_last_error() returns the text for the
 *     calling thread;
 *   - re-entrant; no global mutable state apart from the thread-local error string.
 */
#ifndef STP3_B200_H_
#define STP3_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STP3_OK 0
#define STP3_EINVAL (-1)   /* bad argument (shape, alignment, null pointer) */
#define STP3_ENOSPC (-2)   /* workspace too small */
#define STP3_ECUDA (-3)    /* CUDA runtime / driver error (launch failure, no device) */
#define STP3_EUNSUPPORTED (-4)

/* Library / build identification ("sm_100a", ABI version). */
int stp3_abi_version(void);
const char* stp3_build_info(void);
const char* stp3_last_error(void);

/* ---------------------------------------------------------------------------------------------------------
 * Lift-splat: softmax(depth) (x) context outer product, ego-motion aligned voxel pooling, temporal discount.
 *
 * Replaces, fused into one scatter kernel + one finalize kernel:
 *   STP3.get_geometry                      stp3/models/stp3.py:186-201   (frustum -> ego points)
 *   STP3.encoder_forward (softmax, outer)  stp3/models/stp3.py:214-221   (never materialised)
 *   STP3.projection_to_birds_eye_view      stp3/models/stp3.py:226-301   (ego warp, voxel index, mask, pooling,
 *                                                                          discount recurrence, (C,X,Y) layout)
 *   VoxelsSumming.forward                  stp3/utils/geometry.py:299-318
 *
 * Layouts (all fp32 unless noted)
 *   feat          feat_layout==0: (B,S,N,C,Hf,Wf)  [the reference Encoder's NCHW output]
 *                 feat_layout==1: (B,S,N,Hf,Wf,C)  [channels-last, produced by this library's conv kernels]
 *   depth_logits  (B,S,N,D,Hf,Wf); ignored (may be NULL) when use_depth_distribution==0 (stp3.py:218)
 *   cam_M         (B,S,N,3,3) = R . K^-1   evaluated on the host with the reference's torch calls
 *   cam_t         (B,S,N,3)
 *   ego_R, ego_t  (B,S,3,3), (B,S,3)  from pose_vec2mat(future_egomotion)  (geometry.py:158-172)
 *   xs, ys, ds    (Wf), (Hf), (D): the three axes of STP3.create_frustum (stp3.py:111-130)
 *   bev_off       HOST float[3] = (bev_start_position - bev_resolution/2) as evaluated in fp32 by torch (stp3.py:288)
 *   bev_res       HOST float[3]
 *   ranks_out     optional (B,S,N,D,Hf,Wf) int32: pillar rank ix*(ny*nz)+iy*nz+iz of every lifted point after the
 *                 ego warp, -1 where the reference's mask (stp3.py:239-246) drops it.  Bit-exact with the CPU
 *                 reference; used by the parity tests.
 *   out           out_layout==0: (B,S,C,nx,ny) fp32  [what projection_to_birds_eye_view returns]
 *                 out_layout==1: (B,S,nx,ny,C) fp32  [channels-last]
 *                 out_layout==2: two bf16 planes [2][B,S,nx,ny,C] (hi then lo; C % 8 == 0): the activation format
 *                                of the tensor-core path, consumed directly by stp3_conv_fwd
 *   pool_sum      optional (B,S,C) fp32: sum over the nx*ny cells of out[b,t,c] (feeds the pyramid-pooling branch
 *                 of TemporalBlock, temporal.py:408-423); fully overwritten by the call.
 *   workspace     >= stp3_lift_splat_workspace_bytes(...) bytes, 256-byte aligned.  It holds the channels-last
 *                 fp32 scatter grid (B,S,nx*ny,C) and a per-pillar occupancy map.  It must be ALL ZERO on entry:
 *                 clear it once with stp3_lift_splat_workspace_init() after allocating it; every successful
 *                 stp3_lift_splat_fwd leaves it zero again (the finalize kernel re-zeroes exactly the pillars it
 *                 read), so no per-call memset is needed.  After a failed call, re-initialise it.
 * nz must be 1 (the reference's squeeze(0) at stp3.py:298 assumes it).
 */
size_t stp3_lift_splat_workspace_bytes(int B, int S, int C, int nx, int ny);
int stp3_lift_splat_workspace_init(void* workspace, size_t workspace_bytes, void* stream);

int stp3_lift_splat_fwd(const float* feat, int feat_layout, const float* depth_logits,
                        const float* cam_M, const float* cam_t, const float* ego_R, const float* ego_t,
                        const float* xs, const float* ys, const float* ds,
                        const float* bev_off /*host[3]*/, const float* bev_res /*host[3]*/,
                        int nx, int ny, int nz, float discount,
                        int B, int S, int N, int D, int Hf, int Wf, int C,
                        int use_depth_distribution,
                        int32_t* ranks_out, float* pool_sum,
                        void* workspace, size_t workspace_bytes,
                        float* out, int out_layout, void* stream);

/* Backward of stp3_lift_splat_fwd (training through the drop-in, SURVEY.md row f2): given grad_out = dLoss/d out
 * (B,S,C,nx,ny) fp32 it returns grad_feat (B,S,N,C,Hf,Wf) and grad_depth_logits (B,S,N,D,Hf,Wf; may be NULL, and is not
 * written when use_depth_distribution == 0).  Replaces the autograd chain of the reference:
 *   VoxelsSumming.backward                 stp3/utils/geometry.py:321-330  (every point receives its pillar's gradient)
 *   projection_to_birds_eye_view           stp3/models/stp3.py:239-296     (mask, index_put, bev = bev*discount + tmp)
 *   outer product + softmax over depth     stp3/models/stp3.py:214-216
 * Voxel indices are recomputed with the forward's exact arithmetic (not differentiable, like the reference's .long()).
 * feat is NCHW (feat_layout 0).  scratch: stp3_lift_splat_bwd_scratch_bytes() bytes of device memory (no invariant).
 * Gathers only, no atomics: deterministic. */
size_t stp3_lift_splat_bwd_scratch_bytes(int B, int S, int C, int nx, int ny);
int stp3_lift_splat_bwd(const float* grad_out, const float* feat, const float* depth_logits,
                        const float* cam_M, const float* cam_t, const float* ego_R, const float* ego_t,
                        const float* xs, const float* ys, const float* ds,
                        const float* bev_off /*host[3]*/, const float* bev_res /*host[3]*/,
                        int nx, int ny, int nz, float discount,
                        int B, int S, int N, int D, int Hf, int Wf, int C, int use_depth_distribution,
                        void* scratch, size_t scratch_bytes, float* grad_feat, float* grad_depth_logits, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Dense layers: implicit-GEMM convolution on tcgen05 tensor cores (TMEM accumulators, TMA-fed operands).
 *
 * One entry point covers every convolution of the temporal block, the per-frame DeepLab head and the BEV decoder:
 *   CausalConv3d / conv_1x1x1_norm_activated / TemporalBlock   stp3/layers/temporal.py:252-273, 315-325, 426-489
 *   ASPP / DeepLabHead / UpsamplingAdd / UpsamplingConcat      stp3/layers/convolutions.py:183-280
 *   Decoder (ResNet-18 stages + heads)                         stp3/models/decoder.py:8-140
 * Eval-mode BatchNorm is folded into w / bias by the caller (stp3_b200/dense.py); ReLU, residual add, per-image
 * bias (the spatially constant pyramid-pool / ASPP-pool / ego-motion branches) and the concat offset are fused.
 *
 * Activations are channels-last and carried as TWO bf16 planes (hi = bf16(x), lo = bf16(x - hi)) so that the bf16
 * tensor pipe reproduces fp32 convolution to ~1e-5 (three MMAs per product: hi*hi + hi*lo + lo*hi):
 *   x_hi, x_lo   (B, T, H, W, in_cstride) bf16, in_cstride % 64 == 0, padding channels zero
 *   w            [ntaps][cin/64][2 planes][bn][64] bf16: tap-major, K-major rows of 64 input channels
 *   bias         [bn] fp32;  img_bias  optional [B*T][bn] fp32: per-image bias table that REPLACES bias (it must
 *                already contain it): the spatially constant branches and the ego-motion channels enter here
 *   res_hi/lo    optional residual (B*T, Ho, Wo, res_cstride), channels [res_coff, res_coff+bn)
 *   y_hi, y_lo   optional output planes (B*T, Ho, Wo, out_cstride), channels [out_coff, out_coff+bn)
 *   y_f32        optional (B*T, n_valid, Ho, Wo) fp32 in the reference's NCHW layout (final logits), or channels-last
 *                (desc.f32_layout = 1)
 * taps[i] = (dt, dy, dx): input coordinate = output coordinate * stride + d (dt is not strided); coordinates
 * outside the tensor read as zero (this is the reference's zero / causal padding).
 */
typedef struct stp3_conv_desc {
  int B, T, H, W;        /* B samples x T frames are processed; the input tensor is (B, T_total, H, W, in_cstride) */
  int T_total, t0;       /* frames [t0, t0+T) of each sample are processed (T_total = 0 means T_total = T, t0 = 0);
                            outputs / residual / img_bias are indexed by the B*T processed images */
  int in_cstride;        /* channels of the input tensor */
  int cin_off, cin;      /* channel window this convolution reads (multiples of 64) */
  int Ho, Wo;            /* output spatial size */
  int stride;            /* spatial stride, 1 or 2 */
  int ntaps;             /* 1 .. 49 */
  signed char taps[49][3];
  int bn;                /* padded output channels: 64, 128 or 256 */
  int out_cstride, out_coff;
  int n_store;           /* output channels actually stored to y_hi/y_lo (multiple of 8, 0 = bn): lets several
                            convolutions write adjacent windows of one concat tensor */
  int relu;              /* apply ReLU */
  int res_mode;          /* 0 none, 1 residual added before the activation, 2 after it */
  int res_cstride, res_coff;
  int n_valid;           /* real output channels written to y_f32 */
  int sigmoid;           /* apply a sigmoid to y_f32 (instance_center head, decoder.py:70) */
  int tune_n_sub;        /* 0 = automatic; 1 / 2 = sub-tiles (8x16 pixels each) per CTA tile; 3 = 16x16 tile of a CTA pair (cta_group::2);
                            4 / 5 = linear tiling: 128 consecutive output pixels of the flattened (image, oy, ox) space per
                            CTA / 256 per CTA pair, one im2col load per tap, bn = 256 in ONE launch.  Linear tiling takes
                            2-D taps (dt = 0) over every frame (t0 = 0, T = T_total) and no col_sums, head, img_bias or
                            y_f32 (STP3_EINVAL otherwise) */
  int tune_group;        /* 0 = automatic; 1 = never share an activation load between the dy taps of a 3x3; 3 = share;
                            +4 = stream the weights through the smem ring even if they would fit (more activation stages);
                            +8 = (bn 64) one stacked [W_hi; W_lo] operand: 2 MMAs per product instead of 3 */
  int n_cols;            /* output columns that carry weights (0 = bn): rows [n_cols, bn) of every weight block and the
                            bias are zero padding, so the kernel neither loads nor multiplies them (bn <= 128) */
  /* optional (bn = 64): col_sums[img][c] = sum over the output pixels of the activated output (fp32, (B*T, 64)) -- the
     spatial sums the next block's pooling branches need, produced by the epilogue instead of a separate pass.
     col_sums_scratch: stp3_conv_col_sums_scratch_bytes(B*T, 64) bytes of device scratch. */
  float* col_sums;
  float* col_sums_scratch;
  size_t col_sums_scratch_bytes;
  /* optional second destination (bn = 128, plain hi/lo outputs, n_store <= 64): output columns [64, 64 + n_store2) are
     written to y2 (channels [out2_coff, out2_coff + n_store2)) with activation relu2, columns [0, n_store) to y with
     `relu` -- two 64-column convolutions of the same input as ONE launch that reads the input once. */
  void* y2_hi;
  void* y2_lo;
  int out2_cstride, out2_coff, n_store2, relu2;
  /* input channels [k_lo, k_hi) of the window carry data (multiples of 16; k_hi = 0: the whole window): the weights of
     the other channels are zero, so their UMMA K steps are not issued.  k_lo must lie in the first 64-channel block and
     k_hi in the last (narrow convolutions: 35 -> 35 channels of temporal.py:436-461 run 3 of 4 K steps, 32 -> 32 run 2). */
  int k_lo, k_hi;
  int f32_layout;        /* layout of y_f32: 0 = (B*T, n_valid, Ho, Wo) like the reference, 1 = channels-last (B*T, Ho, Wo,
                            n_valid) -- what stp3_lift_splat_fwd(feat_layout = 1) fetches as ONE TMA box per tile (the encoder
                            heads hand their context features over this way, encoder.py:88-95 -> stp3.py:216) */
} stp3_conv_desc;

/* Optional fused 1x1 "head" evaluated on the activated output tile while it is still in registers:
 *   out_k[img, y, x] = b[k] + sum_c w[k][c] * y[img, y, x, c]      (k < n_out <= 8; sigmoid where the mask bit is set)
 * This is the 3x3 conv -> BN -> ReLU -> 1x1 conv(+bias) tail of every decoder head (decoder.py:38-89); several heads
 * that share their input run as ONE convolution (their 3x3 kernels concatenated along N) and each head's 1x1 weights
 * occupy its column block of w.  out[k] points at the (Ho, Wo) fp32 plane of output k for image 0 and consecutive
 * images are img_stride[k] elements apart, so every head writes its own contiguous (n_img, k_out, Ho, Wo) tensor. */
typedef struct stp3_conv_head {
  int n_out;
  const float* w;          /* [n_out][bn] fp32 (device) */
  const float* b;          /* [n_out] fp32 (device) */
  float* out[8];
  long long img_stride[8];
  int sigmoid_mask;
} stp3_conv_head;

/* bytes of device scratch stp3_conv_desc.col_sums needs for n_img images */
size_t stp3_conv_col_sums_scratch_bytes(int n_img, int bn);
int stp3_conv_fwd(const stp3_conv_desc* desc, const void* x_hi, const void* x_lo, const void* w, const float* bias,
                  const float* img_bias, const void* res_hi, const void* res_lo, void* y_hi, void* y_lo,
                  float* y_f32, const stp3_conv_head* head /* may be NULL */, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * ASPP branches + projection of a DeepLabHead as ONE back-to-back tensor-core kernel (stp3/layers/convolutions.py:242-270):
 *   y = relu(BN(project.0(cat_b relu(BN(conv_b(x))))))   for the spatial branches b (1x1 and the dilated 3x3s); the
 * global-pool branch is spatially constant and enters through img_bias like in stp3_conv_fwd.  The 4 x 128-channel concat
 * tensor never exists: every branch's activated 16x16x128 tile is converted to bf16 hi/lo planes in shared memory and
 * multiplied with its slice of the projection weights while the next branch's convolution runs.  hidden = 128 channels.
 *   x_hi, x_lo  (B, T, H, W, in_cstride) bf16 planes, channels [0, cin) read
 *   w           bf16 rows of 64 (K-major), blocks of [hi: 128 rows][lo: 128 rows]:
 *               first one block per (tap of branch 0.., K block of cin) -- BN folded, rows = hidden channels --
 *               then two per branch for the projection (rows = output channels, K = the branch's hidden channels 0..63, 64..127)
 *   br_bias     [n_br][128] fp32 folded BN shifts of the branches;  img_bias [B*T][128] fp32 projection bias table
 *   y_hi, y_lo  (B*T, H, W, out_cstride) bf16 planes, channels [out_coff, out_coff + 128) written
 */
typedef struct stp3_aspp_desc {
  int B, T, H, W;
  int in_cstride, cin;
  int n_br;                   /* 1 .. 4 spatial branches */
  int n_taps[4];              /* 1 .. 9 each; every branch must contain its centre tap (0, 0) */
  signed char taps[4][9][2];  /* (dy, dx) input offsets */
  int out_cstride, out_coff;
  int no_relu;                /* 0: ReLU on the projection output (ASPP); 1: none (3x3 conv -> 1x1 classifier tail) */
  int n_store;                /* output channels written: 128 (0 = default) or 64 (projection rows 64.. are zero padding) */
} stp3_aspp_desc;
int stp3_aspp_fused_fwd(const stp3_aspp_desc* desc, const void* x_hi, const void* x_lo, const void* w,
                        const float* br_bias, const float* img_bias, void* y_hi, void* y_lo, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Tail of a TemporalBlock (stp3/layers/temporal.py:426-489) as ONE back-to-back tensor-core kernel:
 *   out = relu(BN(aggregation 1x1x1 of [path 0 | path 1 | path 2 | pyramid pooling])) + (projection(x) | x)
 * with path 0 / 1 = the causal (2,3,3) / (1,3,3) convolutions of the entry convolutions' outputs `mid` and path 2 = a
 * 1x1x1 convolution of x.  Up to three MMA chains accumulate the paths side by side in TMEM, the activated concat is
 * converted to bf16 hi/lo in shared memory and multiplied with the aggregation weights; the 128-channel concat tensor
 * never exists.  Applicable when every path has <= 48 channels, x <= 64 spatial channels and the block <= 64 outputs.
 *   chain: src (0 = mid, 1 = x), cin_off (64-channel K block read), taps (dt, dy, dx), n_mma (MMA width, multiple of 16),
 *          tmem_col (column of its first output in the hidden accumulator, multiple of 16), [k_lo, k_hi) channels with data
 *   piece_col[pp]: hidden-accumulator column of the 8-channel piece pp of the 128-channel operand P (-1 = zeros)
 *   w: bf16 rows of 64, blocks of [hi: 128 rows][lo: 128 rows]; one block per tap of chain 0, 1, 2, then two blocks of the
 *      aggregation weights (K blocks of P), then one of the projection; output channel n of an N-wide chain sits in row
 *      n (n < N/2) or 64 + n - N/2 (the two CTAs of a pair each load 64 rows)
 *   hid_bias [B*T][128] (P order), img_bias [B*T][64] (aggregation bias + pooling branch), res_bias [B*T][64] or NULL
 *   col_sums optional (B*T, 64): per-image sums over pixels of the output; scratch: stp3_block_fused_scratch_bytes(B*T)
 */
typedef struct stp3_block_chain {
  int src, cin_off, n_taps;
  signed char taps[18][3];
  int n_mma, tmem_col, k_lo, k_hi;
} stp3_block_chain;
typedef struct stp3_block_desc {
  int B, T, H, W;
  int mid_cstride, x_cstride, out_cstride;
  int n_chain;
  stp3_block_chain chain[3];
  int has_res_proj;           /* 1: residual = 1x1 projection of x (chain `res`, 64 outputs); 0: residual = x itself */
  stp3_block_chain res;
  int piece_col[16];
} stp3_block_desc;
size_t stp3_block_fused_scratch_bytes(int n_img);
int stp3_block_fused_fwd(const stp3_block_desc* desc, const void* mid_hi, const void* mid_lo, const void* x_hi,
                         const void* x_lo, const void* w, const float* hid_bias, const float* img_bias,
                         const float* res_bias, void* y_hi, void* y_lo, float* col_sums, void* scratch,
                         size_t scratch_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Memory-bound helpers of the dense path (all tensors channels-last bf16 hi/lo planes unless noted).
 */
/* fp32 (n_img,C,H,W) [channels_last=0, the reference's NCHW] or (n_img,H,W,C) [1] -> hi/lo (n_img,H,W,cp), padding 0.
 * Used where a foreign fp32 tensor enters a drop-in module (e.g. TemporalModel.forward, temporal_model.py:50). */
int stp3_f32_to_hilo(const float* x, int channels_last, int n_img, int C, int H, int W, int cp, void* hi, void* lo,
                     void* stream);
/* hi/lo (n_img,H,W,cstride) channels [c_off, c_off+C) -> fp32 (n_img,C,H,W): module outputs in the reference layout */
int stp3_hilo_to_f32(const void* hi, const void* lo, int n_img, int H, int W, int cstride, int c_off, int C, float* out,
                     void* stream);
/* sums[img][c] = sum over the H*W pixels (fp32, (n_img, cstride)); cstride <= 1024 */
int stp3_spatial_sum(const void* hi, const void* lo, int n_img, int HW, int cstride, float* sums, void* stream);
/* Spatially constant branches folded to a per-image bias of the consuming 1x1 convolution:
 *   m[c] = sums[c] * inv_hw for the C - n_const spatial channels, const_vals[img][c - (C - n_const)] for the trailing
 *       n_const spatially constant ones (their mean is the value); temporal != 0: averaged with the previous frame of
 *       the same sample when it exists -- AvgPool3d((2,H,W), padding (1,0,0), count_include_pad=False), temporal.py:397-415
 *   v = relu(W1 m + b1)  (R);   out[img][co] = (accumulate ? out[img][co] : bias ? bias[co] : 0) + sum_r W2[co][r] v[r]
 * Replaces PyramidSpatioTemporalPooling (temporal.py:375-423) and ASPPPooling (convolutions.py:227-239). */
int stp3_pool_bias(const float* sums, int sums_stride, int n_img, int T, int C, float inv_hw, int temporal,
                   const float* const_vals, int n_const, const float* W1, const float* b1, int R, const float* W2, int CO,
                   const float* bias, float* out, int co_stride, int accumulate, void* stream);
/* y[n][co] = (accumulate ? y[n][co] : bias ? bias[co] : 0) + sum_ci W[co][ci] x[n][ci]: the 6 broadcast ego-motion
 * channels of stp3.py:145-152 as a per-image bias */
int stp3_small_linear(const float* x, const float* W, int n, int ci, int co, const float* bias, float* y, int co_stride,
                      int accumulate, void* stream);
/* y[..., y_coff:y_coff+C] = bilinear_x2(x[..., :C]) (+ skip[..., s_coff:s_coff+C] when skip is given); x is
 * (n_img,h,w,.), skip and y are (n_img,2h,2w,.).  UpsamplingAdd tail (convolutions.py:204-215) and the upsample +
 * concat of UpsamplingConcat (convolutions.py:183-201). */
int stp3_upsample2x_add(const void* x_hi, const void* x_lo, int n_img, int h, int w, int x_cstride, const void* s_hi,
                        const void* s_lo, int s_cstride, int s_coff, void* y_hi, void* y_lo, int y_cstride, int y_coff,
                        int C, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Frame-sharded lift-splat (latency mode, SURVEY.md §8e): when the global batch is smaller than the number of GPUs the
 * B*S camera frames are split across ranks.  Each rank splats its flat frames f_begin + [0, f_count) (f = b*S + t, the
 * ego-motion chain of frame t still uses the poses t..S-2 of its sample) and writes them RAW -- no discount
 * recurrence -- as channels-last fp32 grids out_raw (f_count, nx, ny, C).  After ONE all-gather of those grids
 * (ncclAllGather over NVLink; stp3_b200/parallel.py) every rank holds (B, S, nx, ny, C) and stp3_bev_discount applies
 * out[t] = out[t-1]*discount + raw[t] (stp3.py:296) and emits the bf16 hi/lo planes the temporal block consumes.
 * workspace: stp3_lift_splat_workspace_bytes(f_count, 1, C, nx, ny) bytes, all-zero on entry (same invariant). */
int stp3_lift_splat_frames_fwd(const float* feat, int feat_layout, const float* depth_logits,
                               const float* cam_M, const float* cam_t, const float* ego_R, const float* ego_t,
                               const float* xs, const float* ys, const float* ds,
                               const float* bev_off /*host[3]*/, const float* bev_res /*host[3]*/,
                               int nx, int ny, int nz,
                               int B, int S, int N, int D, int Hf, int Wf, int C,
                               int use_depth_distribution, int f_begin, int f_count,
                               void* workspace, size_t workspace_bytes, float* out_raw, void* stream);
/* The same, FUSED WITH THE ALL-GATHER: the finalize epilogue stores every finished BEV row of flat frame f straight into
 * slot f of all n_peers gathered buffers peer_out[r] (each (B*S, nx, ny, C) fp32; peer-mapped device pointers of every
 * rank's buffer including this rank's own, e.g. from CUDA IPC / torch symmetric memory) over NVLink -- no separate
 * collective launch.  The caller brackets the call with a cross-rank barrier on both sides (buffers free / stores
 * landed) and then runs stp3_bev_discount on its own buffer.  peer_out is a HOST array of n_peers <= 8 pointers. */
int stp3_lift_splat_frames_allgather_fwd(const float* feat, int feat_layout, const float* depth_logits,
                                         const float* cam_M, const float* cam_t, const float* ego_R, const float* ego_t,
                                         const float* xs, const float* ys, const float* ds,
                                         const float* bev_off /*host[3]*/, const float* bev_res /*host[3]*/,
                                         int nx, int ny, int nz,
                                         int B, int S, int N, int D, int Hf, int Wf, int C,
                                         int use_depth_distribution, int f_begin, int f_count,
                                         void* workspace, size_t workspace_bytes,
                                         int n_peers, void* const* peer_out, void* stream);
int stp3_bev_discount(const float* raw /*(B,S,nx,ny,C) fp32*/, int B, int S, int nx, int ny, int C, float discount,
                      void* out_hi, void* out_lo /*(B,S,nx,ny,C) bf16 each*/, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* STP3_B200_H_ */
