/*
 * aae_b200.h -- C ABI of the B200-native Augmented-Autoencoder hot path.
 *
 * The reference (DLR-RM/AugmentedAutoencoder) has no FFI: its device boundary is
 * `tf.Session.run` on a TensorFlow graph (SURVEY.md section 8b).  Each entry point below
 * replaces the TensorFlow sub-graph named in its comment; paths are relative to
 * /root/reference.  The Python classes in augmentedautoencoder_b200/ae/ keep the
 * reference's class/method surface and bind these symbols through ctypes
 * (see INTEGRATION.md for the binding a reference maintainer would add).
 *
 * Conventions
 *   - plain C types only; every pointer named *_dev is a CUDA device pointer on the
 *     handle's device; pointers named *_any may be host or device (copied with
 *     cudaMemcpyDefault); `stream` is a cudaStream_t passed as void*.
 *   - every function returns 0 on success, a negative aae_status otherwise, never throws
 *     and never aborts.  aae_last_error_string() describes the last failure on the
 *     calling thread.
 *   - handles are re-entrant per (handle, stream): no global mutable state; a handle owns
 *     its weights, packed operand copies and a private workspace sized by max_batch.
 *   - tensor layouts follow the reference: activations NHWC float32, conv kernels HWIO,
 *     dense kernels [in,out], crops BGR uint8 or float32 in [0,1]
 *     (auto_pose/ae/ae_factory.py:133, auto_pose/ae/encoder.py:43-66).
 */
#ifndef AAE_B200_H_
#define AAE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define AAE_API __declspec(dllexport)
#else
#define AAE_API __attribute__((visibility("default")))
#endif

typedef enum {
  AAE_OK = 0,
  AAE_ERR_INVALID_ARG = -1,
  AAE_ERR_CUDA = -2,
  AAE_ERR_UNSUPPORTED = -3,
  AAE_ERR_NO_DEVICE = -4,
  AAE_ERR_OOM = -5
} aae_status;

/* Arithmetic used for the dense contractions (convs, dense layers, codebook scores).
 *   AAE_PREC_FP32_SIMT : IEEE fp32 FMA chains on the CUDA cores (exact-order reference path)
 *   AAE_PREC_TC_SPLIT  : tcgen05 tensor cores, every fp32 operand split into two fp16 terms
 *                        (hi + 2^-11 lo), three products hi*hi + hi*lo + lo*hi accumulated in
 *                        fp32 TMEM -- fp32-grade results at tensor-core rate. */
typedef enum { AAE_PREC_FP32_SIMT = 0, AAE_PREC_TC_SPLIT = 1 } aae_precision;

#define AAE_MAX_LAYERS 8

/* Network geometry: the values `build_encoder` / `build_decoder` read from the training cfg
 * (auto_pose/ae/ae_factory.py:33-71; template auto_pose/ae/cfg/train_template.cfg:5-9,44-55). */
typedef struct {
  int32_t in_h, in_w, in_c;            /* H, W, C of the crop: 128,128,3                          */
  int32_t num_layers;                  /* len(NUM_FILTER)                                          */
  int32_t filters[AAE_MAX_LAYERS];     /* NUM_FILTER  (encoder order; the decoder reverses it)     */
  int32_t strides[AAE_MAX_LAYERS];     /* STRIDES                                                  */
  int32_t kernel_size;                 /* KERNEL_SIZE_ENCODER / KERNEL_SIZE_DECODER                */
  int32_t latent;                      /* LATENT_SPACE_SIZE                                        */
  int32_t max_batch;                   /* workspace is sized for this many crops per call          */
  int32_t precision;                   /* aae_precision                                            */
} aae_net_cfg;

typedef struct aae_encoder aae_encoder;
typedef struct aae_decoder aae_decoder;
typedef struct aae_codebook aae_codebook;
typedef struct aae_trainer aae_trainer;
typedef struct aae_mesh aae_mesh;

AAE_API int aae_version(void);
AAE_API const char* aae_last_error_string(void);
/* 1 if a tcgen05-capable device (compute capability 10.x) is present on `device`, else 0. */
AAE_API int aae_device_supported(int device);
/* Total number of CUDA kernels this library has launched in the process (for launch accounting in benchmarks). */
AAE_API int64_t aae_launch_count(void);

/* ---------------------------------------------------------------- Encoder ------------------
 * Replaces Encoder.encoder_out + Encoder.z: 4x [conv5x5 / stride 2 / TF-SAME(1,2) + bias + ReLU],
 * flatten (h,w,c), dense -> latent  (auto_pose/ae/encoder.py:37-68). */
AAE_API int aae_encoder_create(int device, const aae_net_cfg* cfg, aae_encoder** out);
AAE_API int aae_encoder_destroy(aae_encoder* h);
/* layer in [0,num_layers) = conv kernels HWIO [k,k,cin,cout] + bias [cout];
 * layer == num_layers = dense kernel [flat,latent] + bias [latent]  (variable layouts of
 * auto_pose/ae/encoder.py:43-50,62-66 as stored in the TF checkpoint). */
AAE_API int aae_encoder_set_weights(aae_encoder* h, int layer, const float* kernel_any, const float* bias_any, void* stream);
AAE_API int aae_encoder_get_weights(aae_encoder* h, int layer, float* kernel_any, float* bias_any, void* stream);
/* crops NHWC uint8 [B,H,W,C]; the x/255. of auto_pose/ae/codebook.py:58-59 is fused (true fp32 divide). */
AAE_API int aae_encoder_forward_u8(aae_encoder* h, const uint8_t* crops_dev, int batch, float* z_out_dev, void* stream);
/* crops NHWC float32 in [0,1] (the placeholder of auto_pose/ae/ae_factory.py:133). */
AAE_API int aae_encoder_forward_f32(aae_encoder* h, const float* crops_dev, int batch, float* z_out_dev, void* stream);
/* Run-time range guard of AAE_PREC_TC_SPLIT.  The tensor-core path stores activations as 16*x and weights as 256*w in fp16
 * (hi, lo) pairs, i.e. it needs |activation| < 4094 and |weight| < 255.9 -- true for every trained AAE we know of, but not a
 * law.  A value outside that range is never turned into inf/garbage silently: the kernels record it, aae_*_set_weights
 * fails with AAE_ERR_UNSUPPORTED when a weight is out of range, and this call (which synchronises `stream`) reports -- and
 * clears -- an activation overflow of any forward / training step launched on the handle so far, naming the layers in
 * aae_last_error_string().  The forward entry points stay asynchronous; callers that read results on the host
 * (Session.run, Codebook.nearest_rotation) call this after their own synchronisation.  AAE_PREC_FP32_SIMT handles have no
 * such limit and always return AAE_OK.  (The reference's fp32 TF graph has no counterpart: auto_pose/ae/encoder.py:37-68.) */
AAE_API int aae_encoder_range_status(aae_encoder* h, void* stream);
/* Device address of the guard's 32-bit word (NULL for AAE_PREC_FP32_SIMT handles): streaming callers copy it to pinned host
 * memory behind their own results on their own stream and call aae_encoder_range_status only when it is non-zero, so the
 * pipeline is never synchronised for the check (Codebook.nearest_rotation_async). */
AAE_API int aae_encoder_range_word(aae_encoder* h, const uint32_t** word_dev);
/* Device pointer + element count of the activation of conv layer `layer` (NHWC fp32) from the last
 * forward; layer == num_layers gives the flattened encoder_out.  For tests and for the trainer. */
AAE_API int aae_encoder_activation(aae_encoder* h, int layer, const float** ptr_dev, int64_t* count);

/* Device-side stage timing for benchmarks: `enable` switches cudaEvent bracketing of the stages of the NEXT forward calls
 * on/off; if stage_ms_out != NULL the stage durations of the LAST profiled forward are written first (conv layers in
 * order, then the dense layer) and their count is returned (>= 0; negative = error). */
AAE_API int aae_encoder_profile(aae_encoder* h, int enable, float* stage_ms_out, int capacity);

/* ---------------------------------------------------------------- Codebook -----------------
 * Replaces the Codebook graph: tf.nn.l2_normalize(z,1), matmul(zq, embedding_normalized^T),
 * argmax (auto_pose/ae/codebook.py:27,50-51) and the host-side np.argmax / strided argmax /
 * argpartition of Codebook.nearest_rotation (auto_pose/ae/codebook.py:63-71). */
/* embedding_any: [n_rows, latent] float32, rows already L2-normalised (codebook.py:213-216).
 * row_offset: global index of row 0 (non-zero when this handle holds one shard of a row-sharded
 * codebook); reported indices are global. */
AAE_API int aae_codebook_create(int device, const float* embedding_any, int64_t n_rows, int latent, int num_cyclo,
                                int64_t row_offset, int max_batch, int precision, aae_codebook** out);
AAE_API int aae_codebook_destroy(aae_codebook* h);
/* zq = z * rsqrt(max(sum z^2, 1e-12))  (codebook.py:27). */
AAE_API int aae_l2_normalize(const float* z_dev, int batch, int latent, float* zq_out_dev, void* stream);
/* Fused normalise + score + top-k: for every query the k best rows, scores descending, ties broken
 * towards the LOWEST index (np.argmax semantics, codebook.py:64-68).  upright != 0 restricts the
 * search to rows with (global index % num_cyclo) == 0 (codebook.py:66).  The [B,N] cosine matrix is
 * never materialised.  scores_out_dev [B,k] float32, idx_out_dev [B,k] int32 (global row index). */
AAE_API int aae_codebook_match(aae_codebook* h, const float* z_dev, int batch, int k, int upright,
                               float* scores_out_dev, int32_t* idx_out_dev, void* stream);
/* Full cosine matrix [B, n_rows] = `session.run(codebook.cos_similarity)` (codebook.py:50,63). */
AAE_API int aae_codebook_cosine(aae_codebook* h, const float* z_dev, int batch, float* cos_out_dev, void* stream);
/* Merge per-shard top-k lists (all-gathered over NCCL by the host): in [n_shards,B,k] -> out [B,k];
 * equal scores resolve to the lowest global index, so the result is bit-identical to the
 * unsharded match. */
AAE_API int aae_topk_merge(const float* scores_dev, const int32_t* idx_dev, int n_shards, int batch, int k,
                           float* scores_out_dev, int32_t* idx_out_dev, void* stream);
/* Same merge for the single-collective exchange: every rank's match writes its scores and indices into ONE buffer
 * [2][B][k] (plane 0 float32 scores, plane 1 int32 global indices -- 8 bytes per (query, k)), one NCCL all-gather
 * concatenates them to packed_dev = [n_shards][2][B][k].  Halves the collective count of the row-sharded path, whose
 * whole cost is collective latency (SURVEY.md 8e row 3; no reference counterpart: codebook.py:63-71 is single-device). */
AAE_API int aae_topk_merge_packed(const void* packed_dev, int n_shards, int batch, int k,
                                  float* scores_out_dev, int32_t* idx_out_dev, void* stream);
AAE_API int64_t aae_codebook_rows(const aae_codebook* h);
/* Measurement aid: launches a kernel shaped like the fused match (one CTA per SM, the same 193 KB of dynamic shared memory, with
 * with_tmem != 0 the same 512-column TMEM allocation) that does no work -- the fixed launch / carveout / allocation cost that every
 * event-timed or ncu-timed figure of that kernel contains (scripts/match_bench.py --floor). */
AAE_API int aae_launch_floor_probe(int device, int with_tmem, void* stream);
/* Same contract as aae_encoder_profile; one stage: the whole fused match (k = 1). */
AAE_API int aae_codebook_profile(aae_codebook* h, int enable, float* stage_ms_out, int capacity);

/* ---------------------------------------------------------------- Decoder + loss -----------
 * Replaces Decoder.x: dense latent->8*8*512 + ReLU, 3x [NN-resize x2, conv5x5 s1 + ReLU],
 * NN-resize x2, conv5x5 -> C + sigmoid (auto_pose/ae/decoder.py:36-84). */
AAE_API int aae_decoder_create(int device, const aae_net_cfg* cfg, aae_decoder** out);
AAE_API int aae_decoder_destroy(aae_decoder* h);
/* layer 0 = dense_1 [latent, h0*w0*f0]; layers 1..num_layers = the convs in forward order. */
AAE_API int aae_decoder_set_weights(aae_decoder* h, int layer, const float* kernel_any, const float* bias_any, void* stream);
AAE_API int aae_decoder_get_weights(aae_decoder* h, int layer, float* kernel_any, float* bias_any, void* stream);
AAE_API int aae_decoder_forward(aae_decoder* h, const float* z_dev, int batch, float* x_out_dev, void* stream);
/* Same contract as aae_encoder_range_status for the decoder (dense_1 counts as layer 0; the latent fed to the decoder is
 * covered too). */
AAE_API int aae_decoder_range_status(aae_decoder* h, void* stream);
/* Bootstrapped L2 (LOSS: L2, BOOTSTRAP_RATIO r): per-sample top-k of the flattened squared error,
 * k = numel/r, mean over the [B,k] survivors (auto_pose/ae/decoder.py:90-101).
 * grad_out_dev (optional, [B,numel]) receives dLoss/dx. */
AAE_API int aae_bootstrap_l2_loss(const float* x_dev, const float* target_dev, int batch, int numel_per_sample,
                                  int bootstrap_ratio, float* loss_out_dev, float* grad_out_dev, void* stream);

/* ---------------------------------------------------------------- Training input pipeline ---
 * Dataset.batch on the device (auto_pose/ae/dataset.py:456-495): x[mask] = bg[mask], then the imgaug chain of the training
 * cfg (auto_pose/ae/cfg/train_template.cfg:26-37) with every random draw made by the caller:
 *   geom_dev   [B][4 + 2W + 2H] int32 per image: flags (1 affine, 2 coarse dropout, 4 blur), dropout keep bits (low, high
 *              32 bits over the low_h x low_w cells, row-major), 0, then cv2.warpAffine's fixed-point tables adelta[W],
 *              bdelta[W], X0[H], Y0[H] (10 fractional bits, rounding offset included)
 *   lut_dev    [B][C][256] uint8: the composed Add / Invert / Multiply / Multiply / ContrastNormalization table
 *   bilinear_tab_dev [1024][4] uint16: OpenCV's INTER_LINEAR weight table (rows sum to 32768);  row_cell_dev [H] / col_cell_dev [W]: cv2.resize
 *              INTER_NEAREST index maps of the dropout mask;  blur_kernel_q8: 5 host ints summing to 256 (NULL: no blur);
 *   u8_to_float_dev [256]: value / 255.  tmp_dev: [B,H,W,C] uint8 scratch.  out_u8_dev / out_f32_dev: either may be NULL. */
AAE_API int aae_augment_batch(const uint8_t* x_dev, const uint8_t* mask_dev, const uint8_t* bg_dev, int batch, int h, int w, int c,
                              const int32_t* geom_dev, const uint8_t* lut_dev, const uint16_t* bilinear_tab_dev,
                              const uint8_t* row_cell_dev, const uint8_t* col_cell_dev, int low_w, const int32_t* blur_kernel_q8,
                              const float* u8_to_float_dev, uint8_t* tmp_dev, uint8_t* out_u8_dev, float* out_f32_dev, void* stream);

/* ---------------------------------------------------------------- Training step ------------
 * Replaces sess.run(train_op): encoder fwd, decoder fwd, bootstrapped L2, backward, TF-Adam
 * (auto_pose/ae/ae_train.py:128, auto_pose/ae/ae_factory.py:79-95).
 * The arithmetic follows the handles: encoder and decoder must have been created with the same
 * aae_precision.  AAE_PREC_FP32_SIMT runs every contraction as fp32 FMA chains; AAE_PREC_TC_SPLIT
 * runs the forward pass, the data gradients and the weight gradients of all convs with Cin >= 128
 * as tcgen05 GEMMs (split-fp16 x3, gradients re-scaled per tensor and per step by a power of two),
 * the two dense layers and conv1's weight gradient as fp32 kernels; parameters, Adam state and
 * the gradients returned by aae_trainer_get_grads are fp32 in the reference layouts either way. */
AAE_API int aae_trainer_create(aae_encoder* enc, aae_decoder* dec, int bootstrap_ratio, float learning_rate,
                               float beta1, float beta2, float epsilon, aae_trainer** out);
AAE_API int aae_trainer_destroy(aae_trainer* h);
/* x (augmented input) and y (reconstruction target) NHWC float32 [B,H,W,C]; loss_out_dev: 1 float. */
AAE_API int aae_train_step(aae_trainer* h, const float* x_dev, const float* y_dev, int batch, float* loss_out_dev, void* stream);
/* forward + backward only (no parameter update); gradients stay in the trainer. */
AAE_API int aae_trainer_forward_backward(aae_trainer* h, const float* x_dev, const float* y_dev, int batch, float* loss_out_dev, void* stream);
/* which: 0 = encoder, 1 = decoder; layer as in *_set_weights. */
AAE_API int aae_trainer_get_grads(aae_trainer* h, int which, int layer, float* kernel_grad_any, float* bias_grad_any, void* stream);
AAE_API int64_t aae_trainer_global_step(const aae_trainer* h);
/* Optimizer state, so that a training run can be resumed from a checkpoint the way tf.train.Saver does (the reference's
 * Saver stores every variable's Adam slots and the beta powers: auto_pose/ae/ae_train.py:82,111-115).  which / layer as in
 * aae_trainer_get_grads; *_m = first moment (TF slot name "<var>/Adam"), *_v = second moment ("<var>/Adam_1"), same shapes
 * as the variable; NULL pointers are skipped.  aae_trainer_set_global_step(h, n) makes the next update the (n+1)-th
 * (bias correction with beta^(n+1), TF's beta1_power / beta2_power after n steps). */
AAE_API int aae_trainer_get_state(aae_trainer* h, int which, int layer, float* kernel_m_any, float* kernel_v_any, float* bias_m_any,
                                  float* bias_v_any, void* stream);
AAE_API int aae_trainer_set_state(aae_trainer* h, int which, int layer, const float* kernel_m_any, const float* kernel_v_any,
                                  const float* bias_m_any, const float* bias_v_any, void* stream);
AAE_API int aae_trainer_set_global_step(aae_trainer* h, int64_t step);
/* Per-phase device time of the last training step (cudaEvents on the launching stream; tensor-core trainer only):
 * phase_ms_out[0..6] = operand packs, forward + loss, wgrad GEMMs, dgrad GEMMs, glue (masks / bias sums / re-splits),
 * fp32 backward of the dense layers and of conv1, Adam.  Same enable/read contract as aae_encoder_profile; returns the
 * number of values written (0 when nothing was recorded).  Measurement aid for bench.py --workload train. */
AAE_API int aae_trainer_profile(aae_trainer* h, int enable, float* phase_ms_out, int capacity);

/* ---------------------------------------------------------------- Crop extraction ----------
 * Batched AePoseEstimator.extract_square_patch(black_borders=True) + cv2.resize(INTER_LINEAR)
 * (auto_pose/m3_interface/ae_pose_estimator.py:106-131,157-162): one launch for all detections of a frame, bit-exact
 * with OpenCV's 8-bit fixed-point path.  image_dev: BGR uint8 [img_h, img_w, 3]; boxes_xywh_dev: [n,4] float32 pixel
 * boxes (truncated to int like the reference); out_dev: NHWC uint8 [n, out_size, out_size, 3]. */
AAE_API int aae_extract_square_patches(const uint8_t* image_dev, int img_h, int img_w, const float* boxes_xywh_dev,
                                       int n_boxes, float pad_factor, int out_size, uint8_t* out_dev, void* stream);

/* ---------------------------------------------------------------- Mesh renderer ------------
 * Batched rasteriser of the reference's phong renderer (auto_pose/meshrenderer/meshrenderer_phong.py, shader
 * depth_shader_phong.{vs,frag}; MODEL: reconst, ANTIALIASING: 1).  DESIGN.md "Renderer" states the contract and the fp32
 * operation order.  vertices: host float32 [n_vertices, 9] = position * vertex_scale, normal, colour / 255;
 * faces: host int32 [n_faces, 3], drawn in this order (equal depth: the earlier triangle wins).
 * views_dev: float32 [n_views, AAE_RENDER_VIEW_FLOATS] per view: [0:16] view matrix (row-major, the camera's T_view_world),
 * [16:32] projection (T_proj_view), [32:48] transpose(inverse(view)), [48:54] light 0 = (x, y, z, ambient, diffuse,
 * specular) in eye coordinates, [54:60] light 1, [60:64] unused.
 * workspace_dev: at least aae_render_workspace_bytes(mesh, n_views, W, H) bytes of device memory.
 * flags_dev: int32 [n_views], AAE_RENDER_* bits; a view with AAE_RENDER_BEHIND_CAMERA (a vertex at camera z <= near) is
 * not rasterised.  obj_bb_dev: int32 [n_views, 4] = calc_2d_bbox of the covered pixels (x, y, w, h). */
#define AAE_RENDER_VIEW_FLOATS 64
#define AAE_RENDER_BEHIND_CAMERA 1
#define AAE_RENDER_EMPTY 2
#define AAE_RENDER_BAD_CROP 4
AAE_API int aae_mesh_create(int device, const float* vertices, int64_t n_vertices, const int32_t* faces, int64_t n_faces,
                            aae_mesh** out);
AAE_API int aae_mesh_destroy(aae_mesh* h);
AAE_API int64_t aae_render_workspace_bytes(const aae_mesh* h, int n_views, int W, int H);
/* Full frames with light 0: bgr_dev uint8 [n, H, W, 3] (BGR, row 0 = top), depth_dev float32 [n, H, W] (camera z, 0 where
 * nothing was drawn). */
AAE_API int aae_render_frames(const aae_mesh* h, const float* views_dev, int n_views, int W, int H, float near_plane,
                              float far_plane, void* workspace_dev, int64_t workspace_bytes, uint8_t* bgr_dev, float* depth_dev,
                              int32_t* obj_bb_dev, int32_t* flags_dev, void* stream);
/* Square crops without materialising the frames (Dataset.extract_square_patch + cv2.resize INTER_NEAREST of the frame):
 * crop_x_dev uint8 [n, out_h, out_w, 3] with light 0 around obj_bb shifted by offsets_dev[v] * (w, h) (float64 [n, 2], NULL:
 * no shift); mask_x_dev uint8 [n, out_h, out_w] = 1 where crop x shows no object (NULL: not written); crop_y_dev (NULL: not
 * written) with light 1 around the unshifted obj_bb.  col_map_dev int32 [W + 1, out_w] / row_map_dev int32 [H + 1, out_h]:
 * row s is the INTER_NEAREST source index of every output column / row for a source of size s. */
AAE_API int aae_render_crops(const aae_mesh* h, const float* views_dev, int n_views, int W, int H, float near_plane,
                             float far_plane, const double* offsets_dev, double pad_factor, int out_h, int out_w,
                             const int32_t* col_map_dev, const int32_t* row_map_dev, void* workspace_dev, int64_t workspace_bytes,
                             uint8_t* crop_x_dev, uint8_t* mask_x_dev, uint8_t* crop_y_dev, int32_t* obj_bb_dev, int32_t* flags_dev,
                             void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AAE_B200_H_ */
