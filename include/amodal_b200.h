/* amodal_b200.h -- C ABI of libamodal_b200.so: the B200 (sm_100a) implementation of the discriminative forward pass of
 * Amodal-Depth-Anything (guided Depth-Anything-V2).
 *
 * The reference has no FFI of its own; its boundary for this path is the Python class
 *   AmodalDAv2.forward(x, guide_rgb, guide_mask, observation)      src/models/amodalsynthdrive/dav2.py:64-85
 *   DepthAnythingV2.forward(x, guidance_mask)                      .../depth_anything_v2/dpt.py:225-231
 * Every entry point below names the reference code it replaces. All pointers are plain device (or, where stated, host)
 * pointers; no torch types cross this boundary. Functions return 0 on success and a negative ADA_E* code on failure;
 * ada_last_error() returns a thread-local human readable reason. Nothing throws across the ABI.
 * There is no CPU fallback: compute entry points fail with ADA_ENODEVICE when no sm_100 device is usable.
 */
#ifndef AMODAL_B200_H
#define AMODAL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ADA_OK 0
#define ADA_EINVAL (-1)     /* bad argument / unknown weight key / wrong shape */
#define ADA_ENODEVICE (-2)  /* no CUDA device, or device is not sm_100 */
#define ADA_ECUDA (-3)      /* a CUDA call or kernel failed; see ada_last_error() */
#define ADA_ESTATE (-4)     /* called in the wrong order (e.g. forward before finalize) */

typedef struct ada_model* ada_handle;

/* Architecture description == the constructor arguments of DepthAnythingV2 (dpt.py:201-223) + DINOv2() (dinov2.py:430-448). */
typedef struct ada_config {
  int32_t embed_dim;         /* 384 / 768 / 1024 / 1536                      dinov2.py:370-420 */
  int32_t depth;             /* 12 / 12 / 24 / 40 */
  int32_t num_heads;         /* embed_dim / 64 */
  int32_t ffn_kind;          /* 0 = Mlp fc1-GELU-fc2 (mlp.py:35-41), 1 = SwiGLUFFNFused (swiglu_ffn.py:29-33,45-63) */
  int32_t ffn_hidden;        /* 4*embed_dim (Mlp) or 4096 (SwiGLU @1536) */
  int32_t taps[4];           /* intermediate_layer_idx                       dpt.py:213-218 */
  int32_t features;          /* DPT feature width F                          dav2.py:32-34 */
  int32_t out_channels[4];   /* reassemble widths C_i                        dav2.py:32-34 */
  int32_t guide_channels;    /* channels of patch_embed_guidance (0 = 'none') dinov2.py:110-125 */
  int32_t sigmoid;           /* final activation of output_conv2: 1 = Sigmoid (dpt.py:146-151), 0 = none ('ssi' in
                                loss_stategy, dpt.py:138-144), 2 = ReLU (un-guided model, depth_anything_v2_raw/dpt.py:109-116,182) */
  int32_t pos_grid;          /* sqrt(num_patches) of pos_embed = 37          dinov2.py:437 */
  float interpolate_offset;  /* 0.1                                          dinov2.py:446 */
  int32_t input_projection;  /* 1 = guided head: conv3x3 + channel LN + ReLU per level (dpt.py:153-159,178-179);
                                0 = un-guided DepthAnythingV2 head (depth_anything_v2_raw/dpt.py:118-151) */
  int32_t normalize_input;   /* 1 = rgb in [0,1], ImageNet (x-mean)/std applied inside (dav2.py:65);
                                0 = caller passes the normalised image (depth_anything_v2_raw/dpt.py:168, infer.py:18) */
} ada_config;

/* ---- model lifetime -------------------------------------------------------------------------------------------- */
/* Replaces AmodalDAv2.__init__ / DepthAnythingV2.__init__ (dav2.py:22-61, dpt.py:201-223): creates an empty model. */
int ada_create(const ada_config* cfg, ada_handle* out);
/* Replaces nn.Module.load_state_dict(strict=True) for one tensor: `key` is the reference state-dict name relative to
 * `encoder.` (e.g. "pretrained.blocks.3.attn.qkv.weight", "depth_head.scratch.layer1_rn.weight"); data is fp32,
 * contiguous, host or device memory (copied; the caller keeps ownership). A key that is not part of the architecture
 * described by the config, or a shape that differs from the reference's, fails with ADA_EINVAL (nothing is stored). */
int ada_set_weight(ada_handle h, const char* key, const float* data, const int64_t* shape, int32_t ndim);
/* Packs weights for the kernels: bf16 K-major GEMM operands, fused (3+Cg)-channel patch-embed weight, tap-major conv
 * weights, pre-added biases. Fails with ADA_ESTATE if the state dict is incomplete; ada_last_error() then names every
 * missing key (up to 24 of them, with the total count). */
int ada_finalize(ada_handle h);
/* Replaces AmodalDAv2.forward (dav2.py:64-85) in eval mode. rgb: [B,3,H,W] fp32 in [0,1] (ImageNet normalisation is
 * applied inside, dav2.py:65). guides[i]: [B,guide_ch[i],H,W] fp32, concatenated in order along channels (dav2.py:67-76);
 * sum(guide_ch) must equal cfg.guide_channels. out: [B,1,H,W] fp32. All device pointers, NCHW contiguous.
 * H and W must be multiples of 14 (patch_embed.py:73-74). Asynchronous on `stream` (a cudaStream_t). The call performs no
 * host synchronisation EXCEPT the first time a handle sees a new (B,H,W): the workspace is then re-planned, which drains
 * `stream` first (earlier forwards of this handle may still use the old layout) and may cudaMalloc; the position table of a
 * new patch grid is interpolated on the host once and cached. Steady-state calls at a seen shape are fully asynchronous.
 * Threading: a handle belongs to the device that was current at ada_create and is driven from one thread and one stream
 * at a time (not re-entrant); different handles -- also on different devices of one process -- are independent. */
int ada_forward(ada_handle h, const float* rgb, const float* const* guides, const int32_t* guide_ch, int32_t n_guides,
                float* out, int32_t B, int32_t H, int32_t W, void* stream);
/* Bytes of device workspace the handle holds for its largest (B,H,W) so far. */
size_t ada_workspace_bytes(ada_handle h);
/* Number of kernels the last ada_forward launched (counted while launching; for bench.py's gpu_launches). Pass B = 0 for
 * "whatever the last forward was", or the shape to make sure it is the one meant; 0 if no forward at that shape has run. */
int ada_launch_count(ada_handle h, int32_t B, int32_t H, int32_t W);
/* Test hook: copy a named intermediate of the LAST forward to `dst` (device or host fp32, `count` elements).
 * Names: "tap0".."tap3" ([B,h*w,D] normalised patch tokens, dinov2.py:337-340), "layer1_rn".."layer4_rn",
 * "path_1".."path_4" (NHWC), "tokens" (x after prepare_tokens_with_masks; needs ada_set_capture(h,1)). */
int ada_read_intermediate(ada_handle h, const char* name, float* dst, int64_t count);
int ada_set_capture(ada_handle h, int32_t on);
/* Launch-bound small batches (the reference's infer.py runs one image at a time): when on, the second ada_forward at a
 * given (B,H,W) captures the whole forward into a CUDA graph over handle-owned staging copies of the inputs / output and
 * later calls replay it (3-5 small device copies + one graph launch instead of 136-332 kernel launches). Results are
 * bit-identical to the eager path. Off by default; ignored while profiling / capturing intermediates. */
int ada_set_graph(ada_handle h, int32_t on);
/* Measurement hook (bench.py): when on, every kernel launch of ada_forward is bracketed by CUDA events on the launch
 * stream. ada_profile_read syncs, then sums per kernel class since the last read: elapsed ms, algorithmic FLOPs,
 * algorithmic bytes, launches. Classes: 0 tcgen05 GEMM (linear), 1 tcgen05 GEMM (implicit conv3x3), 2 attention,
 * 3 token LayerNorm, 4 channel LayerNorm+ReLU, 5 bilinear upsample, 6 gathers (patch / cls rows), 7 fused tail
 * gather. n_classes >= 8. */
int ada_set_profile(ada_handle h, int32_t on);
int ada_profile_read(ada_handle h, int32_t n_classes, double* ms, double* flops, double* bytes, int32_t* launches);
/* Raw records since the last ada_profile_read (call before it): meta[5*i..] = class, M, N, K, epi|act<<4|BN<<8; ms[i].
 * Returns the number of records written (<= max_recs) or a negative error code. */
int ada_profile_records(ada_handle h, int32_t max_recs, int32_t* meta, double* ms);
void ada_destroy(ada_handle h);
const char* ada_last_error(void);
/* Device error mailbox written by a kernel that timed out on a barrier (4 words: code, block, parity, thread). */
int ada_device_error(uint32_t out[4]);
/* Bring-up hook: clock64 stamps written by instrumented kernel variants; n <= 512. Only libraries built with
 * -DADA_BRINGUP carry the instrumented kernels (and the ADA_ATT_VARIANT / ADA_GEMM_TIMELINE knobs); the product build
 * returns ADA_ESTATE here. */
int ada_debug_timeline(long long* out, int32_t n);

/* ---- host utility (runs on the CPU; no device needed) -------------------------------------------------------- */
/* Replaces interpolate_pos_encoding (dinov2.py:199-230): bicubic (A=-0.75, align_corners=False, scale_factor =
 * (gh+off)/grid, (gw+off)/grid) resampling of the [grid*grid, D] patch position table to [gh*gw, D]. Host pointers. */
int ada_interp_pos_embed_host(const float* pos_patch, int32_t grid, int32_t D, int32_t gh, int32_t gw, float offset,
                              float* out);

/* The pixel tile an implicit-GEMM 3x3 conv launch (dpt.py:153-159,184-187,193; blocks.py:20-24,57-80) would use for an output
 * map of B x H x W pixels: 2^lw x 2^lh pixels of 2^lb consecutive images (lw + lh + lb = 7, 2 <= 2^lw <= 32), `pair` = 1 single
 * CTA tiles / 2 = two tiles side by side in x (cta_group::2). out = {lw, lh, lb, padded pixels incl. the padding}. The shape
 * is picked for the fewest padded pixels; it depends on the batch, the results do not. Host only. */
int ada_conv_tile_shape(int32_t B, int32_t H, int32_t W, int32_t pair, int64_t out[4]);

/* ---- operator-level entry points (used by tests/ to check each kernel against torch on the same data) --------- */
typedef struct ada_gemm_desc {
  const void* A;        /* bf16 [M,K] row-major (lda) or, conv mode, NHWC [B,H,W,Cin] */
  const void* Bw;       /* bf16 [N,K] row-major (ldb): the torch Linear / packed conv weight */
  int32_t M, N, K, lda, ldb;
  int32_t a_mode;       /* 0 linear, 1 conv3x3 (pad 1; stride 1, or 2 with conv_stride) */
  int32_t epi, act;     /* see EpiMode / ActMode in csrc/gemm.cuh (0 bf16 out, 2 embed, 3 convT, 4 tail, 5 SwiGLU,
                           9 fp32 in-place residual: out_f32 += (acc + bias) * gamma, 10 = mode 0 stored as IEEE fp16) */
  int32_t batch, H, W, Cin;   /* conv mode geometry; EPI_CONVT: input grid */
  const float* bias;
  const float* gamma;
  const float* resid_f32; /* unused (kept for layout stability) */
  float* out_f32;
  void* out_bf16;
  void* out_relu;
  const void* resid1;
  const void* resid2;
  const float* aux;
  int32_t ldo, P, ks, cout, sigmoid;
  int32_t force_bn;     /* 0 = auto, else 32/64/128/256 */
  int32_t force_cg;     /* 0 = auto, 1 = single-CTA tiles, 2 = CTA pairs (tcgen05 cta_group::2) */
  int32_t conv_stride;  /* conv mode: 0 / 1 = stride 1; 2 = stride 2 (resize_layers[3], dpt.py:102-107): H, W describe the
                           INPUT map, the output is ((H-1)/2+1) x ((W-1)/2+1) */
  int32_t conv_taps;    /* conv mode: 0 / 9 = 3x3 taps; 1 = pointwise on 16x8 pixel tiles (Cin % 64 == 0) -- the k == s transposed
                           convs (epi 3) then store their pixel shuffle through TMA boxes (Cout % 64 == 0) */
} ada_gemm_desc;
int ada_op_gemm(const ada_gemm_desc* d, void* stream);
/* out[rows or B*(n_tok-1), D] bf16 = LayerNorm((x + delta) + delta2) (block.py:84,87,105-106; dinov2.py:337-340 when
 * drop_cls). x fp32 [rows, D]; delta / delta2 (optional, bf16 [rows, D]) are the pending residual-branch outputs (delta2
 * requires delta); write_x stores the sum back into x. out2 (optional, with w2 / b2; needs drop_cls == 0): a second affine
 * of the same normalised rows written as the cls-less patch map [B*(n_tok-1), D] -- the tap of a block riding on the next
 * block's norm1 (same input, same statistics; dinov2.py:337-340). */
int ada_op_layernorm(float* x, const void* delta_bf16, const void* delta2_bf16, const float* w, const float* b,
                     void* out_bf16, int32_t rows, int32_t D, float eps, int32_t n_tok, int32_t drop_cls, int32_t write_x,
                     const float* w2, const float* b2, void* out2_bf16, void* stream);
/* ---- single-image pre/post-processing of the reference's infer.py on the device (SURVEY.md section 8 row f2). All
 * pointers are device pointers; one image; asynchronous on `stream`. Nearest sampling follows ATen
 * (src = min(floor(dst * in/out), in-1)), which is what torchvision Resize(NEAREST) and F.interpolate's default use. */
/* uint8 HWC image (cv2 channel order) -> fp32 [3,H,W] in [0,1]: rgb/255 then Resize(NEAREST) (infer.py:84-86);
 * normalize != 0 also applies the ImageNet (x-mean)/std of infer.py:18 (input of the un-guided model). */
int ada_pre_image_nearest(const uint8_t* img_hwc, int32_t H0, int32_t W0, float* out_chw, int32_t H, int32_t W,
                          int32_t normalize, void* stream);
/* uint8 mask (non-zero = inside, infer.py:80-81) -> nearest resize -> mask01 [H,W] in {0,1} (infer.py:87,100-101) and/or
 * the network guide mask01*2-1 (infer.py:91). Either output may be NULL. */
int ada_pre_mask_nearest(const uint8_t* mask, int32_t H0, int32_t W0, float* mask01, float* guide, int32_t H, int32_t W,
                         void* stream);
/* base01 = (d - min d) / (max d - min d) (infer.py:22) and/or observation = base01*2-1 (infer.py:92) over n values;
 * scratch8 = 8 bytes of device memory. Either output may be NULL. */
int ada_post_minmax_normalize(const float* depth, int64_t n, float* base01, float* obs, void* scratch8, void* stream);
/* median_filter_blend(depth_amodal, depth_agg, mask, 3) of infer.py:30-44: out = mask ? amodal : raw, with the seam
 * (3x3 zero-padded mask sum in (0,9)) replaced by the 3x3 box mean of the blended map (cv2.blur, BORDER_REFLECT_101). */
int ada_post_blend_seam(const float* raw01, const float* amodal, const float* mask01, float* out, int32_t H, int32_t W,
                        void* stream);
/* ---- the same pre/post-processing over a batch of B images (B <= 65535), each image's result bit-equal to the
 * single-image entry point's on that image. Images of different sizes live in one packed uint8 device buffer `src`;
 * desc (device, B rows) gives each one's byte offset into it and its size. The rows are read by the kernels, not
 * checked on the host: every image must lie inside `src`. Outputs are dense batches: image b at b * (its per-image
 * size). */
typedef struct ada_img_desc {
  int64_t offset; /* bytes from src to the image's first element */
  int64_t H0, W0; /* its rows and columns (> 0) */
} ada_img_desc;
/* cv2.resize(img, (W, H)) with the default INTER_LINEAR (infer.py:17), bit-exact: uint8 HWC 3-channel images ->
 * out [B,H,W,3] uint8. OpenCV's fixed-point arithmetic (11-bit coefficients); it also equals OpenCV's INTER_AREA path,
 * which cv2 takes when the image is exactly 2H x 2W. An image already H x W comes out unchanged. */
int ada_pre_resize_linear_batch(const uint8_t* src, const ada_img_desc* desc, int32_t B, uint8_t* out_hwc, int32_t H,
                                int32_t W, void* stream);
/* ada_pre_image_nearest per image (3-channel rows of desc) -> out [B,3,H,W]. */
int ada_pre_image_nearest_batch(const uint8_t* src, const ada_img_desc* desc, int32_t B, float* out_chw, int32_t H,
                                int32_t W, int32_t normalize, void* stream);
/* ada_pre_mask_nearest per image (1-channel rows of desc) -> mask01 / guide [B,H,W]; either may be NULL. */
int ada_pre_mask_nearest_batch(const uint8_t* src, const ada_img_desc* desc, int32_t B, float* mask01, float* guide,
                               int32_t H, int32_t W, void* stream);
/* ada_post_minmax_normalize on each of B maps of n values (depth [B,n]), min and max per map; scratch = 8*B bytes of
 * device memory. */
int ada_post_minmax_normalize_batch(const float* depth, int32_t B, int64_t n, float* base01, float* obs, void* scratch,
                                    void* stream);
/* ada_post_blend_seam on each of B maps: raw01, amodal, mask01, out [B,H,W]. */
int ada_post_blend_seam_batch(const float* raw01, const float* amodal, const float* mask01, float* out, int32_t B,
                              int32_t H, int32_t W, void* stream);
/* ---- the pre/post-processing of DepthAnythingV2.infer_image (depth_anything_v2_raw/dpt.py:186-222) over a batch.
 * image2tensor, bit-exact: uint8 BGR HWC images (3-channel rows of desc) -> cvtColor(BGR -> RGB) / 255.0 ->
 * cv2.resize(..., INTER_CUBIC) in float64 -> ImageNet (x - mean) / std in float64 -> out [B,3,H,W] fp32. */
int ada_pre_resize_cubic_normalize_batch(const uint8_t* src, const ada_img_desc* desc, int32_t B, float* out_chw,
                                         int32_t H, int32_t W, void* stream);
/* F.interpolate(depth[:, None], (h, w), mode="bilinear", align_corners=True) of each map of depth [B,H,W] fp32 to its own
 * size: row b of out_desc (device) gives map b's output (h, w) = (H0, W0) and its byte offset from `out` (a multiple of
 * 4). ATen's index math, every operation rounded on its own. */
int ada_post_upsample_restore_batch(const float* depth, int32_t B, int32_t H, int32_t W, const ada_img_desc* out_desc,
                                    float* out, void* stream);
/* ---- per-sample evaluation post-ops of the validation loop on the device (SURVEY.md section 8 row f3;
 * discriminative_trainer.py:542-613). pred [h,w] is resized to the ground-truth size (H,W) by nearest sampling (:542),
 * aligned to depth_obs over visible_mask by least squares (src/util/alignment.py:7-54) and scored against depth_gt + 1e-5
 * over object_mask with the ten metrics of src/util/metric.py:37-161, for the raw and the aligned prediction (:584-613).
 * out24 (device doubles): [0] scale, [1] shift, [2..11] metrics of pred, [12..21] metrics of the aligned prediction in the
 * order abs_relative_difference, squared_relative_difference, rmse_linear, rmse_log, log10, delta1_acc, delta2_acc,
 * delta3_acc, i_rmse, silog_rmse; [22] visible pixels, [23] object pixels. Masks: uint8. scratch26 (26 device doubles) is
 * checked for NULL but no longer written. Runs ada_eval_batch's kernel on one sample: the row is bit-equal to that
 * sample's row in any batch, and the same on every run. */
int ada_eval_sample(const float* pred, int32_t h, int32_t w, const float* depth_gt, const float* depth_obs,
                    const uint8_t* visible_mask, const uint8_t* object_mask, int32_t H, int32_t W, double* out24,
                    double* scratch26, void* stream);
/* ada_eval_sample over a batch of B samples (B <= 65535) whose predictions and ground truths each have their own size.
 * desc (device, B rows) locates sample b: its [h,w] prediction at pred + desc[b].pred (elements) and its four [H,W] maps
 * at byte offsets from src (fp32 depth_gt, fp32 depth_obs, uint8 visible and object masks). The rows are read by the
 * kernel, not checked on the host: every map must lie inside its buffer, fp32 maps 4-byte aligned, H*W < 2^31.
 * out: [B,24] device doubles, row b in the out24 layout. Deterministic, no atomics: row b is bit-equal to ada_eval_sample
 * on sample b, whatever the batch and on every run. */
typedef struct ada_eval_desc {
  int64_t pred;                        /* element offset of the sample's [h,w] prediction from `pred` */
  int64_t gt, obs, visible, object;    /* byte offsets from `src` (fp32, fp32, uint8, uint8 maps of [H,W]) */
  int64_t h, w, H, W;
} ada_eval_desc;
int ada_eval_batch(const float* pred, const uint8_t* src, const ada_eval_desc* desc, int32_t B, double* out, void* stream);
/* Dataset means of the validation loop: adds the B rows [B,24] (ada_eval_batch's out) into acc, (n_buckets + 1) x 22 device
 * doubles. Row 0 of acc is "overall", row 1 + k is bucket k; each holds n_used, n_skipped and the sums of the 20 metric
 * values [2..21] of the rows it took. A row with a NaN among its 20 metric values is counted in n_skipped and left out of
 * the sums (discriminative_trainer.py:596-597). bucket (device int32 [B], or NULL for "overall" only) labels the rows; a
 * label outside [0, n_buckets) counts in "overall" only. Rows are added in order, so acc is the same bits however the
 * samples are split into calls. 1 <= B <= 65535, 0 <= n_buckets <= 65535. */
int ada_eval_accumulate(const double* rows, int32_t B, const int32_t* bucket, int32_t n_buckets, double* acc, void* stream);
/* qkv bf16 [B,N,3,heads,64] -> out bf16 [B,N,heads*64] (attention.py:49-62). impl: -1 = the kernel ada_forward would pick for
 * this shape, 0 = attention.cuh (one 128-query tile per CTA), 1 = attention2.cuh (persistent, 256 queries per work unit). */
int ada_op_attention(const void* qkv_bf16, void* out_bf16, int32_t B, int32_t N, int32_t heads, int32_t impl, void* stream);
/* NHWC bf16 channel LayerNorm + ReLU (dpt.py:56-61,156-158). */
int ada_op_channel_ln_relu(const void* in_bf16, const float* w, const float* b, void* out_bf16, int64_t pixels, int32_t C,
                           float eps, void* stream);
/* NHWC bf16 bilinear, align_corners=True (blocks.py:144, dpt.py:194). */
int ada_op_upsample(const void* in_bf16, void* out_bf16, int32_t B, int32_t Hi, int32_t Wi, int32_t Ho, int32_t Wo,
                    int32_t C, void* stream);
/* fp32 NCHW planes -> bf16 patch matrix [B*P, Kpad] (dav2.py:65,73-74 + patch_embed.py:76 im2col-free gather). */
int ada_op_patch_gather(const float* rgb, const float* const* guides, const int32_t* guide_ch, int32_t n_guides,
                        void* out_bf16, int32_t B, int32_t H, int32_t W, int32_t Kpad, void* stream);
/* Fused tail (dpt.py:194-195): V = per-tap 1x1 contractions of output_conv2.0 applied to the low-res output_conv1 map,
 * NHWC fp16 [B,Hl,Wl,288] (ada_op_gemm with epi = 10); out[b,y,x] = sigmoid(w3 . relu(b2 + sum_taps bilinear_align_corners(V_tap)(y+dy, x+dx)) + b3),
 * aux = [w3 (32), b3]. Requires the 8h -> 14h geometry (Hl*14 == H*8). */
int ada_op_tail_gather(const void* v_f16, const float* bias2, const float* aux, float* out, int32_t B, int32_t Hl, int32_t Wl,
                       int32_t H, int32_t W, int32_t sigmoid, void* stream);
/* Tail on tensor cores, one kernel (dpt.py:194-195): l_f16 = the output_conv1 map, NHWC fp16 [B,Hl,Wl,C] (conv with
 * epi = 10); bilinear 8h -> 14h upsample (align_corners), conv3x3(C -> 32) with zero padding as a tcgen05 GEMM over
 * upsampled tiles built in shared memory, ReLU, 1x1 conv, sigmoid (1) / ReLU (2) / nothing (0); out fp32 [B,H,W].
 * wpk_f16 from ada_pack_tail_mma; aux = [w3 (32), b3]. Requires C % 32 == 0, C <= 128, Hl*14 == H*8, W % 14 == 0. */
int ada_op_tail_mma(const void* l_f16, const void* wpk_f16, const float* bias2, const float* aux, float* out, int32_t B,
                    int32_t Hl, int32_t Wl, int32_t H, int32_t W, int32_t C, int32_t sigmoid, void* stream);
/* output_conv2.0 weight [32,C,3,3] (host fp32) -> [ky][C/8][kx*32+co][8] fp16 on the device (288*C elements). */
int ada_pack_tail_mma(const float* w_host, int32_t C, void* dst_dev_f16);
/* output_conv2.0 weight [32,Cm,3,3] (host fp32) -> [(tap*32+co), Cm] bf16 on the device. */
int ada_pack_tail_taps(const float* w_host, int32_t Cm, void* dst_dev_bf16);
/* Weight packers (host fp32 in, device bf16 out) -- the same code ada_finalize uses. */
int ada_pack_conv3x3(const float* w_host, int32_t Cout, int32_t Cin, void* dst_dev_bf16 /* [Cout, 9*round_up(Cin,64)] */);
int ada_pack_convT(const float* w_host, int32_t Cin, int32_t Cout, int32_t ks, void* dst_dev_bf16 /* [ks*ks*Cout, Cin] */);

#ifdef __cplusplus
}
#endif
#endif /* AMODAL_B200_H */
