/* lungmask_b200 — C ABI of the B200-native lungmask hot path.
 *
 * The reference (JoHof/lungmask) is pure Python and has no FFI for this path; the interface each
 * entry point replaces is therefore a Python function of the reference, cited per function
 * (paths relative to the reference root).  The Python shell in lungmask_b200/ binds these with
 * ctypes (INTEGRATION.md shows the stub a maintainer of the reference would add).
 *
 * Conventions: every function returns 0 on success and a non-zero code on failure
 * (lm_last_error() then returns a static, thread-local message); nothing throws.  The caller owns
 * all host buffers; the engine owns all device memory.  One engine drives one CUDA device; calls on
 * one engine must be serialised by the caller.  "dev" variants take device pointers on the engine's
 * device and run on the engine's stream without host copies.
 *
 * Numerics: the convolutions carry every fp32 value as an fp16 pair (hi + lo * 2^-11, 22 significant bits) on the
 * tensor cores and accumulate in fp32; results match the reference's fp32 forward within 1e-4 on the log-softmax
 * scores.  fp16 saturates at 65504: every activation tensor and every layer's weights carry a power-of-two scale
 * (exact: no significand changes); when a value would leave the range the engine lowers that tensor's scale and runs
 * the forward again, transparently.  LM_ERR_RANGE remains only for non-finite weights and for activations beyond
 * about 1e14 - it never returns a silently wrong mask.
 */
#ifndef LUNGMASK_B200_H
#define LUNGMASK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define LM_API __attribute__((visibility("default")))
#else
#define LM_API
#endif

typedef struct lm_engine lm_engine;

#define LM_NET_RES 256           /* mask.py:166: utils.preprocess(..., resolution=[256, 256]) */
#define LM_MAX_SLOTS 4           /* weight slots (e.g. 0 = base model, 1 = fill model) */
#define LM_FLAG_NO_POSTPROCESS 1 /* LMInferer(volume_postprocessing=False), mask.py:191-194 */
#define LM_ERR_RANGE (-40)       /* non-finite weight, or an activation beyond every representable scale (see "Numerics") */

/* Engine lifetime.  Replaces LMInferer.__init__'s device pick + model.to(device), mask.py:118-139.
 * batch_capacity = slices per forward wave (the reference's batch_size only bounds memory, results
 * are per-slice independent; mask.py:172-187). */
LM_API int lm_create(int device, int batch_capacity, lm_engine** out);
LM_API void lm_destroy(lm_engine* e);
LM_API const char* lm_last_error(void);
LM_API int lm_device(const lm_engine* e);
LM_API int lm_batch_capacity(const lm_engine* e);

/* Number of floats lm_load_weights expects for a model with n_classes outputs. */
LM_API size_t lm_weight_blob_floats(int n_classes);

/* Replaces get_model()'s load_state_dict + model.to(device), mask.py:54-68.  `blob` is the live
 * tensors of the reference state_dict, fp32, concatenated in this order:
 *   for each of the 18 conv3x3 layers in execution order
 *     (down_path.{0..4}.block.{0,3}, up_path.{0..3}.conv_block.block.{0,3}):
 *       conv.weight (OIHW), conv.bias, bn.weight, bn.bias, bn.running_mean, bn.running_var
 *   for each up_path.{0..3}.up.1: weight (OI11), bias
 *   last.weight (K,64,1,1), last.bias (K)
 * n_classes = len(last.bias) (mask.py:56). */
LM_API int lm_load_weights(lm_engine* e, int slot, const float* blob, size_t n_floats, int n_classes);

/* LMInferer._inference for numpy input, mask.py:141-210: int16 HU volume (S,H,W) in host memory ->
 * uint8 label volume (S,H,W) in host memory.  flags: LM_FLAG_*. */
LM_API int lm_apply_volume(lm_engine* e, int slot, const int16_t* vol, int S, int H, int W, int flags, uint8_t* out);
/* Same with device-resident input and output (no host<->device copies). */
LM_API int lm_apply_volume_dev(lm_engine* e, int slot, const int16_t* d_vol, int S, int H, int W, int flags, uint8_t* d_out);

/* LMInferer.apply with a fill model, mask.py:223-232 (two inferences + spare-label fusion +
 * postprocessing(spare=[max+1]) at the original resolution).  flags: LM_FLAG_NO_POSTPROCESS reaches the two inner
 * _inference calls only (mask.py:191-194 honours volume_postprocessing there); the fusion post-processing of
 * mask.py:232 is unconditional, exactly as in the reference. */
LM_API int lm_apply_fused(lm_engine* e, int slot_base, int slot_fill, const int16_t* vol, int S, int H, int W, int flags,
                          uint8_t* out);
/* Same with a device-resident input volume and output (no host<->device copies). */
LM_API int lm_apply_fused_dev(lm_engine* e, int slot_base, int slot_fill, const int16_t* d_vol, int S, int H, int W, int flags,
                              uint8_t* d_out);
/* The fusion glue alone, mask.py:228-230: spare = res_l.max() + 1 (uint8 arithmetic); res_l[(res_l == 0) & (res_r > 0)]
 * = spare; res_l[res_r == 0] = 0.  Host (S,H,W) uint8 in, fused (S,H,W) uint8 + the spare value out (parity tap: the
 * array utils.postprocessing(res_l, spare=[spare]) receives at mask.py:232). */
LM_API int lm_fuse(lm_engine* e, const uint8_t* res_l, const uint8_t* res_r, int S, int H, int W, uint8_t* fused,
                   int* spare_value);

/* LMInferer.apply for FLOAT volumes (float32, or float64 with is_f64 != 0), slot_fill >= 0 for the fusion.  The
 * reference keeps the input dtype through utils.preprocess (clip and bilinear zoom without rounding, utils.py:44-45,
 * 108-110) and normalises in that dtype (mask.py:167-168) before the cast to fp32 (mask.py:178-182); so does the engine. */
LM_API int lm_apply_volume_float(lm_engine* e, int slot, int slot_fill, const void* vol, int is_f64, int S, int H, int W,
                                 int flags, uint8_t* out);
/* utils.preprocess(resolution=[256,256]) + the normalisation of mask.py:167-168 for a float volume: the fp32 network
 * input (S,256,256) and the crop boxes (parity tap). */
LM_API int lm_preprocess_float(lm_engine* e, const void* vol, int is_f64, int S, int H, int W, float* normalised,
                               int32_t* boxes);

/* LMInferer.apply for a SimpleITK image, mask.py:157-164,204-208,223-232: the array `vol` (n0,n1,n2) is in the image's
 * NATIVE orientation; lps = transpose(vol, perm) flipped along every axis k with flip[k] != 0 is the array of the image
 * re-oriented to DICOM "LPS" (lungmask_b200/orient.py derives perm / flip from the direction cosines).  The engine
 * re-orients on the device, runs the path on the LPS array and returns the mask in the native orientation (n0,n1,n2).
 * slot_fill >= 0 selects the fusion of mask.py:223-232, whose spare-label fusion and post-processing run on the
 * native-orientation results exactly as in the reference (each _inference call re-orients its own result back). */
LM_API int lm_apply_volume_oriented(lm_engine* e, int slot, int slot_fill, const int16_t* vol, int n0, int n1, int n2,
                                    const int* perm, const int* flip, int flags, uint8_t* out);

/* ---- one volume over several GPUs (SURVEY.md 8e; the reference is single-device, mask.py:118-121) ----------------
 * One process and one engine per GPU.  Slices are independent up to the 3-D post-processing (utils.py:48-51,
 * mask.py:173-187,196-202 vs utils.py:293-358): rank r of `world` runs pre-processing and the network on the contiguous
 * slice range [r * ceil(S/world), (r+1) * ceil(S/world)) and the uint8 argmax volume (plus the crop boxes) is
 * all-gathered once - by the engine itself: every rank owns a gather block in device memory that its peers map through
 * CUDA IPC, a rank pushes its slab into every peer's block over NVLink and raises an epoch flag there; post-processing
 * and reshape then run replicated on the gathered volume and every rank holds the whole result.  The 3-D labelling of
 * utils.py:293 is slab-sharded too: every rank labels its own slices, the union-find parents travel with the labels,
 * and after the gather only the slab boundaries are linked ("shard_slab_ccl", default 1).
 *   lm_shard_init     allocates this rank's gather block for volumes of up to max_slices slices
 *   lm_shard_export   writes the block's IPC handle (lm_shard_handle_bytes() bytes) - exchange it by any host channel
 *   lm_shard_connect  maps the peers' blocks; `handles` = world handles in rank order (this rank's own is ignored)
 *   lm_apply_volume_sharded      every rank passes the SAME (S,H,W) host volume (only its slab is copied to the device)
 *                                and receives the whole (S,H,W) result (out may be NULL on ranks that do not need it)
 *   lm_apply_volume_sharded_dev  device-resident whole-volume buffers on this rank's device (only the slab is read)
 *   lm_shard_labels   parity / alternative-collective tap: device pointers of this rank's gathered boxes (int32 x 4
 *                     per slice) and labels (256*256 bytes per slice), and the slice capacity
 * The calls are collective: every rank must make them in the same order (a bounded device-side wait turns a missing
 * peer into error -50 instead of a hang).  world == 1 needs no export / connect. */
LM_API int lm_shard_init(lm_engine* e, int rank, int world, int max_slices);
LM_API size_t lm_shard_handle_bytes(void);
LM_API int lm_shard_export(lm_engine* e, void* handle_out);
LM_API int lm_shard_connect(lm_engine* e, const void* handles);
LM_API int lm_shard_labels(lm_engine* e, void** d_boxes, void** d_labels, size_t* slice_cap);
LM_API int lm_apply_volume_sharded(lm_engine* e, int slot, const int16_t* vol, int S, int H, int W, int flags, uint8_t* out);
LM_API int lm_apply_volume_sharded_dev(lm_engine* e, int slot, const int16_t* d_vol, int S, int H, int W, int flags,
                                       uint8_t* d_out);

/* ---- compressed DICOM pixel data (what SimpleITK / GDCM decode for utils.read_dicoms, utils.py:186-190) -----------
 * lm_decode_frames decodes n_frames single-component 16-bit frames, each encoded in data[offset, offset + length):
 *   LM_CODEC_JPEG_LOSSLESS  ITU-T T.81 process 14 (SOF3, Huffman): predictors 1-7, point transform, restart intervals
 *                           of whole rows; transfer syntaxes 1.2.840.10008.1.2.4.57 and .4.70
 *   LM_CODEC_RLE            DICOM PS3.5 Annex G (1.2.840.10008.1.2.5): exactly 2 segments, most significant bytes first
 * into out as stored 16-bit values, the frames one after the other (frame i starts at the sum of rows * cols of the
 * frames before it).  With is_signed and a JPEG precision P < 16 the values are sign-extended from bit P - 1.
 * frame_status[i] is 0 or one of LM_ERR_DECODE_* (a failed frame's output is unspecified).  The call returns 0 once
 * every frame has a status, non-zero (lm_last_error) for invalid arguments or a CUDA error.  It needs no engine: it
 * runs on `device` with its own stream and scratch memory, frees both and synchronises before it returns.  All
 * pointers are host pointers. */
#define LM_CODEC_JPEG_LOSSLESS 1
#define LM_CODEC_RLE 2
#define LM_ERR_DECODE_HEADER (-60) /* unsupported or malformed JPEG marker segments (frame type, Nf, size, EOI) or RLE header */
#define LM_ERR_DECODE_DATA (-61)   /* entropy-coded data: undefined Huffman code, unexpected marker, RSTm out of sequence */
#define LM_ERR_DECODE_LENGTH (-62) /* JPEG: a restart interval ends before its samples, or the RSTm count differs from the
                                      * number of intervals (codewords after the last sample are ignored, as libjpeg-turbo
                                      * does); RLE: a segment ends before, or runs past, rows * cols bytes */
typedef struct {
  uint64_t offset, length;
  int32_t codec, rows, cols, is_signed;
} lm_frame;
LM_API int lm_decode_frames(int device, const uint8_t* data, size_t n_bytes, const lm_frame* frames, int n_frames,
                            uint16_t* out, int32_t* frame_status);

/* ---- stage-level entry points (each mirrors one reference function; used by the parity tests) ---- */

/* utils.preprocess(img, resolution=[out_h,out_w]), utils.py:32-52 (+ simple_bodymask :55-82,
 * crop_and_resize :85-111): (S,H,W) int16 -> resized (S,out_h,out_w) int16 + boxes (S,4) int32
 * [r0, c0, r1, c1] half-open.  clip != 0 applies np.clip(-1024, 600) (utils.py:45) as preprocess does;
 * clip == 0 gives utils.crop_and_resize on each slice as-is. */
LM_API int lm_preprocess(lm_engine* e, const int16_t* vol, int S, int H, int W, int out_h, int out_w, int clip,
                         int16_t* resized, int32_t* boxes);
/* utils.simple_bodymask, utils.py:55-82: one slice (H,W) int16 (NOT clipped) -> (H,W) uint8 0/1. */
LM_API int lm_simple_bodymask(lm_engine* e, const int16_t* slice, int H, int W, uint8_t* mask);

/* Normalise + UNet.forward + argmax, mask.py:167-187 / resunet.py:58-70: resized (S,256,256) int16 ->
 * labels (S,256,256) uint8 and, if scores != NULL, the LogSoftmax scores (S,K,256,256) fp32. */
LM_API int lm_forward(lm_engine* e, int slot, const int16_t* resized, int S, uint8_t* labels, float* scores);

/* utils.postprocessing(label_image, spare, skip_below), utils.py:272-358 on a (S,H,W) uint8 volume. */
LM_API int lm_postprocess(lm_engine* e, const uint8_t* labels, int S, int H, int W, const int32_t* spare, int n_spare,
                   int skip_below, uint8_t* out);

/* utils.keep_largest_connected_component(mask), utils.py:390-404: (S,H,W) uint8 0/1 mask -> 0/1 mask of its largest
 * full-connectivity component (ties: the last in raster order).  Fails (like the reference) on an empty mask. */
LM_API int lm_keep_largest_component(lm_engine* e, const uint8_t* mask, int S, int H, int W, uint8_t* out);

/* [utils.reshape_mask(mask[i], boxes[i], (H,W)) for i], utils.py:114-129 + mask.py:196-202:
 * (S,mask_h,mask_w) uint8 + boxes -> (S,H,W) uint8. */
LM_API int lm_reshape_masks(lm_engine* e, const uint8_t* masks, int mask_h, int mask_w, const int32_t* boxes, int S,
                            int H, int W, uint8_t* out);

/* Per-stage device time (ms, CUDA events on the engine stream) of the last lm_apply_volume*:
 * [0] H2D, [1] preprocess, [2] forward, [3] postprocess, [4] reshape, [5] D2H, [6] total.
 * Also the number of kernels the engine launched in that call. */
LM_API int lm_last_timings(const lm_engine* e, float* ms7, int64_t* kernel_launches);

/* Options: "time_convs" (0/1: bracket every tensor-core convolution launch with CUDA events on the engine
 * stream; read the sum with lm_last_conv_timing after an lm_apply_volume* call), "chunk_kb" (k-blocks
 * accumulated inside the tensor core between fp32 round-to-nearest adds; sets both layer classes),
 * "chunk_kb_wide" (the same for the layers with >= 128 output channels only; defaults: 1 for the 64-channel
 * layers, 2 for the wide ones), "dual_issue" (0/1: a second MMA-issuing thread per CTA on alternate chunks;
 * default 0), "cta_pairs" (0/1: the cta_group::2 convolution kernel: validated, on par, default 0),
 * "weight_mcast" (0 / 2: clusters of two CTAs share every weight stage through TMA multicast),
 * "stem_v2" (0 = first stem kernel, 1 = register-resident, 2 = shared-memory tile, 3 = the same with the next tile's
 * samples fetched one tile ahead, the default; all bit-identical),
 * "graphs" (1, default: a volume's forward - every wave's ~26 launches - is captured once as a CUDA graph and replayed;
 * 0: every kernel is launched individually; per-launch convolution timing and score taps always launch individually),
 * "upsample_v2" (0: one thread per output sample, 1: per cell, 2 = default: per cell with static corner indexing; all bit-identical),
 * "merge_ctas" (0, default: the region merge loop of utils.py:310-339 runs on one CTA per SM in batches of independent
 * candidates; 1: the single-CTA sequential loop; n: that many CTAs),
 * "ccl_rule" (1 = pruned neighbour rule of the 26-connected labelling, the default; 0 = probe all 13 backward
 * neighbours), "post_region_capacity" (test hook: size of the post-processing's region tables),
 * "post_debug_stage" (parity taps of the post-processing). */
LM_API int lm_set_option(lm_engine* e, const char* key, int value);
LM_API int lm_last_conv_timing(const lm_engine* e, float* conv_ms, int64_t* conv_launches);

/* Parity taps: intermediate activations of the LAST forward wave, as fp32 [n][H][W][C] (channels last; the
 * hi/lo operand planes are joined).  Activation ids follow the execution order of the network:
 * 0 A0(stem out) 1 S0 2 P0 3 A1 4 S1 5 P1 6 A2 7 S2 8 P2 9 A3 10 S3 11 P3 12 A4 13 B4 (encoder: A = first conv,
 * S = block output / skip, P = pooled) 14 L0 15 U0 16 C0 17 E0 18 L1 19 U1 20 C1 21 E1 22 L2 23 U2 24 C2 25 E2
 * 26 L3 27 U3 28 C3 (decoder: L = 1x1 conv below the upsample, U = upsampled, C = first conv, E = block output). */
LM_API int lm_debug_activation_info(int act_id, int* level, int* channels, int* split);
LM_API int lm_debug_read_activation(lm_engine* e, int act_id, int n, float* out);

/* Forward-only benchmark hook: runs the forward pass on `S` device-resident resized slices and
 * reports the device time of the convolution kernels alone (ms) for the roofline. */
LM_API int lm_forward_dev(lm_engine* e, int slot, const int16_t* d_resized, int S, uint8_t* d_labels, float* conv_ms);

#ifdef __cplusplus
}
#endif
#endif /* LUNGMASK_B200_H */
