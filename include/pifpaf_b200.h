/*
 * pifpaf_b200.h -- C ABI of the B200-native OpenPifPaf inference hot path.
 *
 * Plain C: opaque handles, raw pointers and sizes, int status codes; no C++
 * exceptions cross this boundary and no torch types appear in any signature.
 * Every entry point cites the reference interface it replaces (paths relative
 * to /root/reference/src/openpifpaf/).  The shared library is
 * openpifpaf_b200/csrc/libpifpaf_b200.so (sm_100a only; there is no CPU path:
 * every call fails with PIFPAF_E_CUDA when no B200 is present).
 *
 * Threading: a handle is stateful and not re-entrant (like the reference's
 * CifCaf instance, csrc/include/openpifpaf/decoder/cifcaf.hpp:91-94); use one
 * handle per (GPU, stream) from one host thread at a time.  Configuration is
 * passed BY VALUE per call (the reference keeps process-global statics,
 * csrc/src/module.cpp:26-32,76-117).
 */
#ifndef PIFPAF_B200_H_
#define PIFPAF_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PIFPAF_OK 0
#define PIFPAF_E_BADARG 1     /* TORCH_CHECK-class argument error in the reference */
#define PIFPAF_E_CUDA 2       /* CUDA runtime/driver error (incl. "no device") */
#define PIFPAF_E_OVERFLOW 3   /* a capacity given at create() time was exceeded */
#define PIFPAF_E_NOMEM 4

/* Last error message of the calling thread ("" if none). */
const char* pifpaf_last_error(void);
/* Library/ABI version and build architecture string ("sm_100a"). */
int pifpaf_abi_version(void);
const char* pifpaf_build_arch(void);

/* ------------------------------------------------------------------------ */
/* Decoder configuration: the reference's static knobs, by value.            */
/* Defaults in brackets; citations are the reference definitions.            */
typedef struct pifpaf_decoder_params {
    int64_t cifhr_neighbors;           /* [16]    csrc/src/cif_hr.cpp:13 */
    double cifhr_threshold;            /* [0.3]   csrc/src/cif_hr.cpp:14 */
    int32_t cifhr_ablation_skip;       /* [0]     csrc/src/cif_hr.cpp:15 */
    double seed_threshold;             /* [0.2]   csrc/src/cif_seeds.cpp:11 */
    int32_t seeds_ablation_nms;        /* [0]     csrc/src/cif_seeds.cpp:13 */
    int32_t seeds_ablation_no_rescore; /* [0]     csrc/src/cif_seeds.cpp:14 */
    double caf_score_th;               /* [0.3]   csrc/src/caf_scored.cpp:11 */
    double caf_cif_floor;              /* [0.1]   csrc/src/cifcaf.cpp:153 */
    int32_t caf_ablation_no_rescore;   /* [0]     csrc/src/caf_scored.cpp:12 */
    int32_t block_joints;              /* [0]     csrc/src/cifcaf.cpp:18 (no effect there either) */
    int32_t greedy;                    /* [0]     csrc/src/cifcaf.cpp:19 */
    double keypoint_threshold;         /* [0.15]  csrc/src/cifcaf.cpp:20 */
    double keypoint_threshold_rel;     /* [0.5]   csrc/src/cifcaf.cpp:21 */
    int32_t reverse_match;             /* [1]     csrc/src/cifcaf.cpp:22 */
    int32_t force_complete;            /* [0]     csrc/src/cifcaf.cpp:23 */
    double force_complete_caf_th;      /* [0.001] csrc/src/cifcaf.cpp:24 */
    double nms_suppression;            /* [1e-5]  csrc/src/nms_keypoints.cpp:12 */
    double nms_instance_threshold;     /* [0.15]  csrc/src/nms_keypoints.cpp:13 */
    double nms_keypoint_threshold;     /* [0.15]  csrc/src/nms_keypoints.cpp:14 */
    double occ_reduction;              /* [2.0]   csrc/include/openpifpaf/decoder/cifcaf.hpp:103 */
    double occ_min_scale;              /* [4.0]   same */
    /* CifHr revision the arithmetic is carried out at.  A fresh reference
     * instance decodes at 1.0 (csrc/src/cif_hr.cpp:115); the parity contract is
     * "fresh instance per image", so keep 1.0 unless reproducing a warm one. */
    double cifhr_revision;             /* [1.0] */
} pifpaf_decoder_params_t;

int pifpaf_decoder_default_params(pifpaf_decoder_params_t* params);

/* ------------------------------------------------------------------------ */
/* CifCaf decoder.  Replaces torch.classes.openpifpaf_decoder.CifCaf
 * (csrc/src/module.cpp:24-58; csrc/src/cifcaf.cpp:116-262).                  */
typedef struct pifpaf_decoder pifpaf_decoder_t;

/* CifCaf(n_keypoints, skeleton): csrc/include/openpifpaf/decoder/cifcaf.hpp:96-107.
 * skeleton: [n_connections][2] int64, 0-BASED (the reference's Python passes
 * skeleton-1, decoder/cifcaf.py:119-122).  n_cif_fields normally == n_keypoints.
 * Capacities (no allocation happens on the decode path):
 *   max_batch, max_h, max_w : largest field batch/shape (cells) to be decoded;
 *   max_stride              : largest field stride (hi-res map side = (h-1)*stride+1);
 *   max_annotations         : per-image capacity for annotations before NMS.
 * device: CUDA device ordinal. */
int pifpaf_decoder_create(pifpaf_decoder_t** out, int32_t device,
                          int32_t n_keypoints, int32_t n_cif_fields,
                          int32_t n_connections, const int64_t* skeleton,
                          int32_t max_batch, int32_t max_h, int32_t max_w, int32_t max_stride,
                          int32_t max_annotations);
void pifpaf_decoder_destroy(pifpaf_decoder_t* dec);

/* Batched decode of DEVICE-resident fields (the entry point the reference
 * lacks: decoder/decoder.py:88-100 moves every field to the CPU first).
 *   cif_dev [B][F][5][h][w] f32, caf_dev [B][C][8][h][w] f32, contiguous.
 *   init_ann_dev: optional [B][init_cap][K][4] f32 (v,x,y,s) device pointer with
 *   init_ids_dev [B][init_cap] i64 and init_counts_dev [B] i32, or NULL
 *   (csrc/src/cifcaf.cpp:177-202).
 * All work is enqueued on `stream` (a cudaStream_t); results stay on the device
 * until pifpaf_decoder_fetch(). */
int pifpaf_decoder_decode_device(pifpaf_decoder_t* dec,
                                 const float* cif_dev, const float* caf_dev,
                                 int32_t batch, int32_t h, int32_t w,
                                 int32_t cif_stride, int32_t caf_stride,
                                 const float* init_ann_dev, const int64_t* init_ids_dev,
                                 const int32_t* init_counts_dev, int32_t init_cap,
                                 const pifpaf_decoder_params_t* params, void* stream);

/* Copy the results of the last decode to host buffers and wait for them.
 *   counts [B] i32: annotations per image (after NMS);
 *   ann [B][ann_cap][K][4] f32 (v,x,y,s), ids [B][ann_cap] i64 (-1 unless initial ids).
 * Returns PIFPAF_E_OVERFLOW if any image exceeded max_annotations (pre-NMS) or
 * ann_cap (post-NMS); counts[] then still holds the true post-NMS counts. */
int pifpaf_decoder_fetch(pifpaf_decoder_t* dec, int32_t* counts, float* ann, int64_t* ids,
                         int32_t ann_cap, void* stream);

/* Split fetch for pipelining: fetch_begin enqueues ONE async D2H of the packed results of the last decode
 * (header + up to 512 KB of records) on `stream` and returns at once; fetch_end waits for it and unpacks
 * (same outputs as pifpaf_decoder_fetch).  Results are double buffered: a new decode may be enqueued
 * between begin and end; at most two fetches may be outstanding, completed in order. */
int pifpaf_decoder_fetch_begin(pifpaf_decoder_t* dec, void* stream);
int pifpaf_decoder_fetch_end(pifpaf_decoder_t* dec, int32_t* counts, float* ann, int64_t* ids, int32_t ann_cap);
/* Wait for the oldest outstanding fetch and report its per-image counts without consuming it
 * (lets the caller size the buffers it passes to fetch_end). */
int pifpaf_decoder_fetch_peek(pifpaf_decoder_t* dec, int32_t* counts);

/* Single image, HOST buffers: the call the reference's binding makes.
 * Replaces CifCaf::call / call_with_initial_annotations
 * (csrc/src/cifcaf.cpp:116-262): cif [F][5][h][w], caf [C][8][h][w] on the host;
 * H2D, decode and D2H happen inside.  *n_out receives N; out_ann [cap][K][4],
 * out_ids [cap]. */
int pifpaf_decoder_call(pifpaf_decoder_t* dec,
                        const float* cif, int32_t cif_stride,
                        const float* caf, int32_t caf_stride,
                        int32_t h, int32_t w,
                        const float* initial_annotations, const int64_t* initial_ids, int32_t n_initial,
                        const pifpaf_decoder_params_t* params,
                        float* out_ann, int64_t* out_ids, int32_t cap, int32_t* n_out);

/* Stage taps of the last decode, for parity tests (the reference exposes the
 * same stages through torch.classes.openpifpaf_decoder_utils, module.cpp:66-118).
 * All copy to HOST buffers for image `b` and synchronise.
 *   cifhr  [F][H][W] f32 (CifHr.get_accumulated, csrc/src/cif_hr.cpp:92-94);
 *   seeds  f [n] i64 + vxys [n][4] f32 sorted (CifSeeds.get, csrc/src/cif_seeds.cpp:93-114);
 *   caf    per connection [n][7] f32 (CafScored.get, csrc/src/caf_scored.cpp:86-104):
 *          out_fwd/out_bwd are [C][h*w][7], counts in n_fwd/n_bwd [C]. */
int pifpaf_decoder_tap_cifhr(pifpaf_decoder_t* dec, int32_t b, float* out, int64_t out_elems);
int pifpaf_decoder_tap_seeds(pifpaf_decoder_t* dec, int32_t b, int64_t* out_f, float* out_vxys,
                             int64_t cap, int64_t* n_out);
int pifpaf_decoder_tap_caf(pifpaf_decoder_t* dec, int32_t b, float* out_fwd, int64_t* n_fwd,
                           float* out_bwd, int64_t* n_bwd);

/* Tests only: move the handle's validity tags next to their wrap-around points.  Occupancy::clear and the fresh
 * CifHr buffer of a new reference instance (csrc/src/occupancy.cpp:71-77, csrc/src/cif_hr.cpp:97-121) are epoch
 * tags here (a byte per occupancy cell, a word per CifHr tile); when a tag would wrap the maps are really cleared
 * once.  occupancy_epoch: odd, 1..255 (two tags per decode); cifhr_epoch: any 32-bit value. */
int pifpaf_decoder_debug_set_epochs(pifpaf_decoder_t* dec, uint32_t occupancy_epoch, uint32_t cifhr_epoch);

/* Work counters of the last decode, summed over its batch (synchronises; bench.py's decoder roofline):
 * stats[0] hi-res CifHr pixels written (the map is tile-sparse), [1] seeds (CifSeeds.get), [2] CAF list entries
 * (forward + backward, CafScored.get; of the force-complete refill if that ran), [3] annotations before NMS;
 * with n_stats >= 10 also the seed loop's diagnostics: [4] rounds, [5] seeds grown speculatively, [6..9] SM clocks
 * spent in setup / seed selection / growing / committing (one CTA per image, summed). */
int pifpaf_decoder_last_stats(pifpaf_decoder_t* dec, int64_t* stats, int32_t n_stats);

/* Free op grow_connection_blend (csrc/src/cifcaf.cpp:32-113, module.cpp:60):
 * caf [n][7] f32 HOST; writes x,y,s,v to out_xysv[4]. */
int pifpaf_grow_connection_blend(const float* caf, int64_t n, double x, double y, double s,
                                 double filter_sigmas, int32_t only_max, double* out_xysv);


/* ------------------------------------------------------------------------ */
/* CifDet decoder.  Replaces torch.classes.openpifpaf_decoder.CifDet
 * (csrc/src/cifdet.cpp:24-80, module.cpp:57-62; CifDetHr csrc/src/cif_hr.cpp:124-150, CifDetSeeds
 * csrc/src/cif_seeds.cpp:69-90,117-139) and, with params.nms != 0, the post-processing of the reference's Python
 * wrapper (decoder/cifdet.py:55-64: torchvision batched_nms / nms, score suppression, instance threshold).       */
typedef struct pifpaf_cifdet pifpaf_cifdet_t;

typedef struct {
    int64_t cifhr_neighbors;           /* CifHr::neighbors [16]  csrc/src/cif_hr.cpp:13 */
    double cifhr_threshold;            /* CifHr::threshold [0.3] csrc/src/cif_hr.cpp:14 */
    double seed_threshold;             /* CifDetSeeds::threshold [0.2] csrc/src/cif_seeds.cpp:12 */
    double occ_reduction;              /* Occupancy(2.0, 4.0): include/openpifpaf/decoder/cifdet.hpp:40 */
    double occ_min_scale;
    double cifhr_revision;             /* [1.0] revision of a fresh instance's first call */
    int64_t max_detections_before_nms; /* CifDet::max_detections_before_nms [120] csrc/src/cifdet.cpp:16 */
    int32_t nms;                       /* 0: raw output of CifDet::call; 1: + decoder/cifdet.py:55-64 */
    int32_t nms_by_category;           /* CifDet.nms_by_category [1] decoder/cifdet.py:20 */
    double iou_threshold;              /* [0.5]  decoder/cifdet.py:17 */
    double suppression;                /* [0.1]  decoder/cifdet.py:22 */
    double instance_threshold;         /* [0.15] decoder/cifdet.py:18 */
} pifpaf_cifdet_params_t;

int pifpaf_cifdet_default_params(pifpaf_cifdet_params_t* params);

/* Capacities like pifpaf_decoder_create; max_detections bounds max_detections_before_nms. */
int pifpaf_cifdet_create(pifpaf_cifdet_t** out, int32_t device, int32_t n_categories,
                         int32_t max_batch, int32_t max_h, int32_t max_w, int32_t max_stride,
                         int32_t max_detections);
void pifpaf_cifdet_destroy(pifpaf_cifdet_t* det);

/* Batched decode of DEVICE-resident fields [B][F][6][h][w] f32 (intensity, confidence, x, y, w, h), enqueued on
 * `stream`.  Results stay on the device until pifpaf_cifdet_fetch(). */
int pifpaf_cifdet_decode_device(pifpaf_cifdet_t* det, const float* field_dev, int32_t batch, int32_t h, int32_t w,
                                int32_t stride, const pifpaf_cifdet_params_t* params, void* stream);

/* counts [B]; records [B][cap][8] f32 per detection: category (1-based, as a float), score, x1, y1, x2, y2
 * (csrc/src/cifdet.cpp:61-63), score after NMS suppression, kept flag (1.0 = score after NMS > instance
 * threshold); without params.nms the last two are (score, 1.0).  Synchronises `stream`. */
int pifpaf_cifdet_fetch(pifpaf_cifdet_t* det, int32_t* counts, float* records, int32_t cap, void* stream);

/* Single image, HOST field [F][6][h][w]: the call the reference's binding makes (CifDet::call). */
int pifpaf_cifdet_call(pifpaf_cifdet_t* det, const float* field, int32_t stride, int32_t h, int32_t w,
                       const pifpaf_cifdet_params_t* params, float* records, int32_t cap, int32_t* n_out);


/* ------------------------------------------------------------------------ */
/* Image preprocessing on the GPU.  Replaces, on the inference path of the reference's Predictor
 * (predictor.py:85-102), transforms.RescaleAbsolute(fast=True) -> PIL.Image.resize(BILINEAR)
 * (transforms/scale.py:154-176,56-59) and the image part of transforms.CenterPad / CenterPadTight
 * (transforms/pad.py:15-110).  Raw uint8 HWC images, resized bit-identically to Pillow's ImagingResample
 * (horizontal pass into an 8-bit intermediate, then vertical; 22-bit fixed-point coefficients) straight into a
 * window of a padded canvas [H][W][3] that pifpaf_net_forward_u8 consumes.
 *   xbounds [dst_w][2] / xkk [dst_w][xksize], ybounds [dst_h][2] / ykk [dst_h][yksize]: device int32 tables of
 *   Pillow's precompute_coeffs + normalize_coeffs_8bpc (built by the host mirror, openpifpaf_b200/preprocess.py);
 *   a direction whose size does not change needs none.  tmp: device scratch of src_h * dst_w * 3 bytes.
 *   dst points at the window's first pixel inside the canvas, dst_pitch_bytes = canvas row pitch. */
int pifpaf_image_resize_bilinear_u8(const uint8_t* src_dev, int32_t src_h, int32_t src_w,
                                    uint8_t* dst_dev, int64_t dst_pitch_bytes, int32_t dst_h, int32_t dst_w,
                                    const int32_t* xbounds_dev, const int32_t* xkk_dev, int32_t xksize,
                                    const int32_t* ybounds_dev, const int32_t* ykk_dev, int32_t yksize,
                                    uint8_t* tmp_dev, void* stream);
/* constant RGB fill of a canvas of n_pixels pixels: the pad colour (CenterPad draws a random grey per image,
 * transforms/pad.py:52-54; CenterPadTight uses (124, 116, 104), transforms/pad.py:100-101) */
int pifpaf_image_fill_rgb(uint8_t* dst_dev, int64_t n_pixels, int32_t r, int32_t g, int32_t b, void* stream);


/* ------------------------------------------------------------------------ */
/* Network forward: backbone + CompositeField4 heads (network/nets.py:35-48,
 * network/basenetworks.py:186-355, network/heads.py:272-378), as a list of fused
 * ops over NHWC bf16 activation tensors.  The host mirror of the reference
 * modules (openpifpaf_b200/network.py) walks a Shell-like module, folds
 * BatchNorm (eval) into weights+bias and channel_shuffle/chunk into physical
 * channel placement, and emits these ops once; forward() replays them.
 * All weights are HOST f32 pointers (copied/converted at emit time).
 *
 * Activation codes: the `relu` / `dw_relu` argument of the ops below selects the activation fused into the epilogue,
 * applied in f32 before the bf16 rounding (torchvision MobileNetV2 / V3 blocks, basenetworks.py:407-458):
 *   0 none, 1 ReLU, 2 ReLU6 (torch.nn.ReLU6), 3 Hardswish (torch.nn.Hardswish: x * min(max(x + 3, 0), 6) / 6).
 * Codes 2 and 3 need a 3x3 kernel in pifpaf_net_input_conv; pifpaf_net_dw_conv1x1_scatter accepts 0 and 1 only.                                                            */
typedef struct pifpaf_net pifpaf_net_t;

int pifpaf_net_create(pifpaf_net_t** out, int32_t device, int32_t max_batch);
void pifpaf_net_destroy(pifpaf_net_t* net);

/* Activation tensor NHWC bf16 [max_batch][h][w][c_phys] (zero-initialised;
 * c_phys % 16 == 0: rows start on 32-byte boundaries).  *id receives its handle. */
int pifpaf_net_tensor(pifpaf_net_t* net, int32_t h, int32_t w, int32_t c_phys, int32_t* id);

/* Input block conv (basenetworks.py:275-280; torchvision resnet conv1): dense kxk conv on the
 * f32 NCHW image [B][3][in_h][in_w] -> bf16 NHWC, + bias (folded BN) (+ReLU). weight [c_out][3][k][k]. */
int pifpaf_net_input_conv(pifpaf_net_t* net, int32_t in_h, int32_t in_w, int32_t kernel, int32_t stride,
                          int32_t pad, int32_t c_out, const float* weight, const float* bias,
                          int32_t relu, int32_t out_tensor);

/* 1x1 conv == GEMM on tensor cores (tcgen05, TMA-fed): reads columns [in_col_off, in_col_off+k_cols)
 * of in_tensor; weight [n_out][k_cols] in the same physical column order; + bias (+ReLU).
 * shuffle_src_tensor < 0: plain output at columns [out_col_off, out_col_off+n_out) of out_tensor.
 * shuffle_src_tensor >= 0: fused cat + channel_shuffle(2) (basenetworks.py:233-242): output logical
 *   channel 2n <- shuffle_src[n], 2n+1 <- this conv[n], written contiguously (physical == logical order);
 *   in_col_off must be a multiple of 8 (TMA coordinates must be 16-byte aligned): in the 'shuffle' layout the next
 *   block's x.chunk(2) starts its view at or below n_out on such a column and zeroes the weight columns of the
 *   leading pass-through channels. */
int pifpaf_net_conv1x1(pifpaf_net_t* net, int32_t in_tensor, int32_t in_col_off, int32_t k_cols,
                       int32_t n_out, const float* weight, const float* bias, int32_t relu,
                       int32_t out_tensor, int32_t out_col_off,
                       int32_t shuffle_src_tensor, int32_t shuffle_src_col_off);

/* 1x1 conv whose output columns go to SEVERAL tensors (the 'bins' activation layout of the ShuffleNetV2K stages):
 * torch.cat + channel_shuffle + the next block's x.chunk(2) (basenetworks.py:233-242) only ever move channels, so
 * the host routes every channel, at production time, into the buffer of the block that will consume it
 * (openpifpaf_b200/network.py::_plan_stage_bins) and no pass-through channel is copied.
 * weight [n_out][k_cols] / bias [n_out] are already in GEMM column order (padding columns: zero weight and bias);
 * piece i = GEMM columns [piece_col0[i], +piece_count[i]) -> columns [piece_tensor_col[i], +piece_count[i]) of
 * tensor piece_tensor[i]; pieces tile [0, n_out) in order; counts and tensor columns are multiples of 16
 * (32 bytes: every lane writes whole sectors with 256-bit stores). */
int pifpaf_net_conv1x1_scatter(pifpaf_net_t* net, int32_t in_tensor, int32_t in_col_off, int32_t k_cols,
                               int32_t n_out, const float* weight, const float* bias, int32_t relu,
                               int32_t n_pieces, const int32_t* piece_col0, const int32_t* piece_count,
                               const int32_t* piece_tensor, const int32_t* piece_tensor_col);

/* Dense kxk conv (k <= 7, stride 1 or 2) as an implicit GEMM on tensor cores (torchvision ResNet blocks behind
 * basenetworks.py:71-150): reads channels [in_col_off, in_col_off+c_in) of in_tensor through a 4-D TMA map
 * (zero padding by out-of-bounds fill); weight [n_out][c_in][k][k] (torch layout); + bias (folded BN);
 * optional residual add (residual_tensor >= 0) BEFORE the optional ReLU (BasicBlock / Bottleneck tail). */
int pifpaf_net_conv(pifpaf_net_t* net, int32_t in_tensor, int32_t in_col_off, int32_t c_in,
                    int32_t kernel, int32_t stride, int32_t pad, int32_t n_out, const float* weight,
                    const float* bias, int32_t relu, int32_t out_tensor, int32_t out_col_off,
                    int32_t residual_tensor, int32_t residual_col_off);

/* Depthwise kxk conv (basenetworks.py:228-231), weight [channels][k][k], + bias (folded BN) + activation code.
 * Activation codes 2 and 3 need k = 3 or 5 and stride 1 or 2 (the MobileNet depthwise convs, torchvision
 * InvertedResidual behind basenetworks.py:407-458); 3x3 convs of stride 1 or 2 and every depthwise conv followed
 * by pifpaf_net_se_conv1x1 run on a kernel for any channel count (k_dwconv_nc). */
int pifpaf_net_dwconv(pifpaf_net_t* net, int32_t in_tensor, int32_t in_col_off, int32_t channels,
                      int32_t kernel, int32_t stride, int32_t pad, const float* weight, const float* bias,
                      int32_t relu, int32_t out_tensor, int32_t out_col_off);

/* Squeeze-excitation + linear projection of a MobileNetV3 block (torchvision InvertedResidual with
 * SqueezeExcitation, behind basenetworks.py:432-458): s = Hardsigmoid(fc2(ReLU(fc1(avgpool(x))))), then the 1x1
 * projection conv + folded BN on x * s, no activation, optional residual add (use_res_connect; residual_tensor < 0:
 * none).  in_tensor must be the whole output of the op emitted just before, a pifpaf_net_dwconv over `channels`
 * channels with k = 3 or 5 and stride 1 or 2: that op then also writes per-tile channel sums of its f32 outputs
 * (fixed-order reduction, no atomics: deterministic and independent of the batch).  Emits two ops: a squeeze-excitation
 * kernel (one CTA per image: pooling, fc1, ReLU, fc2, Hardsigmoid) that writes per-image projection weights
 * bf16(weight[n][k] * s[k]), and the projection as the implicit-GEMM conv with kernel 1, each 8 x 16 pixel tile
 * reading the weights of its image.
 * fc1_weight [squeeze][channels], fc1_bias [squeeze], fc2_weight [channels][squeeze], fc2_bias [channels];
 * weight [n_out][channels], bias [n_out]. */
int pifpaf_net_se_conv1x1(pifpaf_net_t* net, int32_t in_tensor, int32_t channels, int32_t squeeze,
                          const float* fc1_weight, const float* fc1_bias, const float* fc2_weight, const float* fc2_bias,
                          int32_t n_out, const float* weight, const float* bias, int32_t out_tensor,
                          int32_t residual_tensor);

/* Depthwise 5x5 (stride 1) -> BatchNorm -> 1x1 conv -> BatchNorm -> ReLU, the tail of InvertedResidualK.branch2
 * (basenetworks.py:219-226), as ONE kernel: the depthwise result is produced tile by tile straight into the
 * shared-memory A operand of the tcgen05 GEMM and never visits HBM.  Arguments: those of pifpaf_net_dwconv
 * (dw_weight [channels][5][5], dw_bias: folded BN) followed by those of pifpaf_net_conv1x1_scatter (weight
 * [n_out][channels] over the depthwise output channels; n_out a multiple of 16, at most 512). */
int pifpaf_net_dw_conv1x1_scatter(pifpaf_net_t* net, int32_t in_tensor, int32_t in_col_off, int32_t channels,
                                  int32_t kernel, int32_t stride, int32_t pad,
                                  const float* dw_weight, const float* dw_bias, int32_t dw_relu,
                                  int32_t n_out, const float* weight, const float* bias, int32_t relu,
                                  int32_t n_pieces, const int32_t* piece_col0, const int32_t* piece_count,
                                  const int32_t* piece_tensor, const int32_t* piece_tensor_col);

/* All CompositeField4 heads as ONE GEMM with the eval epilogue fused (heads.py:330-378):
 * head i has n_fields[i] x n_comp[i] output channels (channel = f*n_comp + comp);
 * comp_ops (concatenated per head, length sum n_comp): 0 raw, 1 sigmoid, 2 +x index, 3 +y index,
 * 4 softplus.  weight [sum n_fields*n_comp][k_cols], bias likewise.
 * Outputs are f32 [B][n_fields][n_comp][h][w] device buffers owned by the net. */
int pifpaf_net_heads(pifpaf_net_t* net, int32_t in_tensor, int32_t k_cols, int32_t n_heads,
                     const int32_t* n_fields, const int32_t* n_comp, const int32_t* comp_ops,
                     const float* weight, const float* bias);
/* The same with `upsample_stride` > 1 heads (heads.py:307-343: the conv emits n_fields*n_comp*up*up channels,
 * torch.nn.PixelShuffle(up) and the crop [ (up-1)/2, size - ceil((up-1)/2) ) follow): the epilogue writes conv
 * channel c*up*up + dy*up + dx of cell (y, x) to output channel c at (y*up + dy - low, x*up + dx - low); index
 * fields are added in the up-sampled grid.  weight [sum n_fields*n_comp*up*up][k_cols].  Outputs
 * [B][n_fields][n_comp][h*up - low - high][w*up - low - high]. */
int pifpaf_net_heads_upsampled(pifpaf_net_t* net, int32_t in_tensor, int32_t k_cols, int32_t n_heads,
                               const int32_t* n_fields, const int32_t* n_comp, const int32_t* comp_ops,
                               int32_t upsample_stride, const float* weight, const float* bias);
int pifpaf_net_head_output(pifpaf_net_t* net, int32_t head, float** dev_ptr,
                           int32_t* n_fields, int32_t* n_comp, int32_t* h, int32_t* w);

/* Head-output buffering.  n_buffers == 2: successive forwards alternate between two sets of head-output buffers, so
 * that the decode of forward i (reading set i & 1 on another stream) may overlap forward i+1;
 * pifpaf_net_head_output then reports the set the LAST forward wrote.  The reference has no counterpart: its fields are
 * fresh tensors per call (network/heads.py:330-378) copied to the host before decoding (decoder/decoder.py:98). */
int pifpaf_net_set_head_buffers(pifpaf_net_t* net, int32_t n_buffers);
/* Cap the persistent grids of the forward kernels at n_sm SMs (0 = all): leaves SMs free for a decode that runs
 * concurrently on another stream (one CTA per image, decoder.cu k_grow). */
int pifpaf_net_set_sm_limit(pifpaf_net_t* net, int32_t n_sm);

/* Shell.forward (network/nets.py:35-48) on images_dev [batch][3][in_h][in_w] f32 (device), async on stream.
 * gemm_impl: 0 = tcgen05 tensor-core kernels (the product); 1 = plain SIMT debug kernel used only
 * by tests to cross-check the tensor-core path. */
int pifpaf_net_forward(pifpaf_net_t* net, const float* images_dev, int32_t batch, int32_t gemm_impl,
                       void* stream);
/* Shell.forward on RAW images: images_nhwc_dev [batch][in_h][in_w][3] uint8 (device).  The stem applies the
 * reference's eval preprocessing on load -- torchvision ToTensor + Normalize (transforms/__init__.py:26-33):
 * ((u / 255) - mean[c]) / std[c], IEEE division and subtraction, zero padding in the normalised domain -- so the
 * fields equal pifpaf_net_forward on the normalised float image bit for bit, with a quarter of the input bytes. */
int pifpaf_net_forward_u8(pifpaf_net_t* net, const uint8_t* images_nhwc_dev, int32_t batch, const float* mean,
                          const float* stdev, int32_t gemm_impl, void* stream);

/* Same as pifpaf_net_forward but brackets every op with CUDA events on `stream` and, after a final
 * synchronise, writes per-op milliseconds to op_ms[num_ops] (profiling leg of bench.py; never the
 * headline timing).  op_kind[i]: 0 input conv, 1 tcgen05 GEMM, 2 depthwise conv, 3 fused depthwise -> GEMM,
 * 4 squeeze-excitation (pifpaf_net_se_conv1x1's first op); op_flops/op_bytes are
 * the algorithmic FLOPs and bytes (inputs + outputs + weights, each once) of op i for this batch. */
int pifpaf_net_forward_timed(pifpaf_net_t* net, const float* images_dev, int32_t batch, int32_t gemm_impl,
                             void* stream, float* op_ms, int32_t* op_kind, double* op_flops, double* op_bytes);
/* Debug/parity tap: copy activation tensor `id` (first `batch` images) to host as f32 [B][h][w][c_phys]. */
int pifpaf_net_tap_tensor(pifpaf_net_t* net, int32_t id, int32_t batch, float* out, int64_t out_elems);
/* Debug/parity: fill activation tensor `id` (first `batch` images) from host f32 [B][h][w][c_phys] (rounded to bf16). */
int pifpaf_net_set_tensor(pifpaf_net_t* net, int32_t id, int32_t batch, const float* data, int64_t n_elems);
/* Algorithmic FLOPs (2*MAC) of one forward per image, and number of ops emitted. */
double pifpaf_net_flops_per_image(pifpaf_net_t* net);
int32_t pifpaf_net_num_ops(pifpaf_net_t* net);

/* Number of kernels this library launched since load (bench.py's gpu_launches). */
int64_t pifpaf_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif  /* PIFPAF_B200_H_ */
