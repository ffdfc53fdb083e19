/* libb200det -- C ABI of the B200-native detect -> embed -> associate hot path.
 *
 * Drop-in boundary for JunweiLiang/Object_Detection_Tracking: the entry points below are what the
 * reference's Python call surface binds for this path (the reference has no native code of its own;
 * its hot path is `sess.run` on a TF graph).  Citations are file:line in the reference repository.
 *
 *   models.get_model(config, gpuid, ...)                       models.py:97-119      -> b2_create + b2_load_weights
 *   model.get_feed_dict_forward(img) + sess.run([final_boxes,
 *       final_labels, final_probs, fpn_box_feat], feed_dict)   obj_detect_tracking.py:610-635,
 *                                                              models.py:1629-1636   -> b2_detect_host / b2_detect
 *   model.get_feed_dict_forward_multi(imgs) + sess.run         models.py:3301-3310,
 *                                                              obj_detect_tracking_multi_queuer.py:474-480 -> same, batch > 1
 *   initialize(load=True, ...) (.npz / ckpt name->array load)  obj_detect_tracking.py:392-448 -> b2_load_weights
 *   NearestNeighborDistanceMetric.distance(features, targets)  deep_sort/nn_matching.py:156-177 -> b2_cosine_cost
 *
 * Conventions: every function returns 0 on success, <0 on error (message via b2_last_error()); no
 * exceptions cross the ABI; plain pointers and sizes only.  A b2_ctx is bound to one device and is
 * single-threaded (the reference calls sess.run from exactly one thread).  The library never
 * allocates caller-visible output memory: callers pass capacity-sized buffers and receive counts.
 */
#ifndef B200DET_H_
#define B200DET_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b2_ctx b2_ctx;

/* Mirrors the fields of the reference's argparse namespace that shape the inference graph
 * (obj_detect_tracking.py:236-389). */
typedef struct b2_config {
  int32_t batch;              /* im_batch_size; frames per b2_detect call */
  int32_t height, width;      /* frame size after resizeImage (nn.py:1540-1560), e.g. 720 x 1280 */
  int32_t input_dtype;        /* 0 = float32 HWC BGR (the reference placeholder), 1 = uint8 HWC BGR */
  int32_t num_class;          /* incl. background (15 ActEV, 81 COCO) */
  int32_t resnet_blocks[4];   /* (3,4,23,3) R101, (3,4,6,3) R50 */
  int32_t use_dilations;      /* --version 3: res5 dilation 2 */
  int32_t class_agnostic;     /* use_frcnn_class_agnostic (versions 4-6) */
  int32_t rpn_topk;           /* rpn_test_post_nms_topk */
  int32_t result_per_im;      /* 100 */
  int32_t fpn_num_channel;    /* 256 */
  int32_t fc_head_dim;        /* 1024 */
  int32_t precision;          /* 0 = fp16 operands / fp32 accumulate; 1 = split fp16 pair (~fp32 products) */
  int32_t conv_impl;          /* 0 = tcgen05 tensor-core kernel, 1 = CUDA-core cross-check kernel */
  int32_t use_cuda_graph;     /* replay the frame as one CUDA graph */
  float max_size;             /* rounded up to a multiple of 32 by the caller */
  float rpn_min_size, rpn_nms_thres, fastrcnn_nms_iou_thres, result_score_thres;
  float anchor_strides[5], anchor_sizes[5], anchor_ratios[3];
  float bbox_reg_weights[4];
  int32_t accum_chunk;        /* split precision: K-blocks (64 elements) the tensor core accumulates before the
                                 partial sum is folded in with round-to-nearest; 0 = default (1), <0 = never */
  int32_t multi_semantics;    /* 1 = post-processing of Mask_RCNN_FPN_multi (combined_non_max_suppression:
                                 no RPN min-size filter, zero-padded level merge + zero-area drop, no score threshold) */
  int32_t add_mask;           /* --add_mask: mask head on the final boxes (models.py:934-961, 1173-1199; mrcnn_head_dim 256):
                                 ROIAlign 14x14 -> 4 x conv3x3 -> 2x2/2 transposed conv -> conv1x1 -> sigmoid of the box's own
                                 class; results through b2_get_masks */
} b2_config;

const char* b2_last_error(void);
int b2_version(void);

int b2_create(b2_ctx** out, int device, const b2_config* cfg);
void b2_destroy(b2_ctx* ctx);

/* Named fp32 host arrays in the reference's Tensorpack-npz naming ("conv0/W",
 * "group1/block0/conv2/bn/mean/EMA", "fpn/lateral_1x1_c2/b", "fastrcnn/fc6/W", ...).
 * BatchNorm is folded, kernels are packed K-major and split into fp16 planes on the device. */
int b2_load_weights(b2_ctx* ctx, const char* const* names, const float* const* data, const int64_t* numel, int n);

/* One pass of the hot path over `batch` frames resident on the device.  All pointers are device
 * pointers; outputs: boxes [B,100,4] x1y1x2y2, probs [B,100], labels [B,100] (1-based), valid [B],
 * box_feat [B*100,C,7,7] fp32 (feat_mode 0) or [B*100,C] mean-pooled (feat_mode 1); any may be NULL.
 * feat_mode 2 / 3 are the TMOT driver's other aggregations (obj_detect_tracking_multi_queuer_tmot.py:511-525): 2 = max over
 * the 7x7 bins [B*100,C], 3 = "spatial" mean over the channels [B*100,49].
 * Asynchronous on the context stream unless `sync` != 0. */
int b2_detect(b2_ctx* ctx, const void* frames_dev, float* boxes, float* probs, int32_t* labels, int32_t* valid,
              float* box_feat, int feat_mode, int sync);
/* Same with host buffers (pinned for full speed): H2D of the frames, the pass, D2H of the results. */
int b2_detect_host(b2_ctx* ctx, const void* frames_host, float* boxes, float* probs, int32_t* labels,
                   int32_t* valid, float* box_feat, int feat_mode);

/* Frame ingest with the resize on the device (SURVEY 8f rank 1).  The reference resizes on the host
 * (frame.astype("float32") -> resizeImage = cv2.resize INTER_LINEAR, nn.py:1540-1560; obj_detect_tracking.py:597-608,
 * enqueuer_thread.py:259-266) and feeds the resized float32 frame.  Here the uint8 source frames [batch, src_h, src_w, 3]
 * (BGR) are uploaded and resized to the context's height x width by a kernel (same bilinear arithmetic, csrc/resize_math.h),
 * then the pass runs as in b2_detect_host.  The context must have input_dtype = 0; the caller picks height / width with
 * get_new_hw (nn.py:1548-1560).  b2_resize_frames runs the resize alone (parity tests), host in / host out. */
int b2_detect_host_resize(b2_ctx* ctx, const uint8_t* frames_u8, int src_h, int src_w, float* boxes, float* probs,
                          int32_t* labels, int32_t* valid, float* box_feat, int feat_mode);
int b2_resize_frames(int device, const uint8_t* frames_u8, int n, int src_h, int src_w, int dst_h, int dst_w,
                     float* out_host);

/* Pipelined ingest for streaming drivers (the queue-fed loop of obj_detect_tracking_multi_queuer.py:386-480):
 * b2_submit_host returns as soon as the upload, the pass and the download of the results are enqueued; b2_wait(slot)
 * blocks until that slot's results are in the caller's buffers.  Two slots: the upload of batch i+1 overlaps the pass
 * of batch i.  Host buffers must stay valid (page-locked for real overlap) until b2_wait returns. */
int b2_submit_host(b2_ctx* ctx, const void* frames_host, float* boxes, float* probs, int32_t* labels, int32_t* valid,
                   float* box_feat, int feat_mode, int slot);
int b2_wait(b2_ctx* ctx, int slot);
/* b2_submit_host for uint8 source frames [batch, src_h, src_w, 3] resized on the device (see b2_detect_host_resize); the
 * source frames must not exceed the network input's float32 byte size (<= 4 source pixels per input pixel). */
int b2_submit_host_resize(b2_ctx* ctx, const uint8_t* frames_u8, int src_h, int src_w, float* boxes, float* probs,
                          int32_t* labels, int32_t* valid, float* box_feat, int feat_mode, int slot);

/* RCNN_FPN_givenbox (models.py:1816-1967, get_model_feat :121-131): final_box_features of GIVEN boxes -- backbone + FPN,
 * ROIAlign 7x7 on the uncropped p2..p5, mean over the bins.  frame_host: one frame of the configured dtype / size (batch 1
 * context), boxes_host [n,4] x1 y1 x2 y2 in frame pixels, feat_host [n, fpn_num_channel]. */
int b2_box_features(b2_ctx* ctx, const void* frame_host, const float* boxes_host, int n, float* feat_host);

/* final_masks of the last pass (needs cfg.add_mask): [batch][result_per_im][28][28] float32 (models.py:958-961; the
 * drivers paste them into the frame with fill_full_mask, obj_detect_tracking.py:719); rows >= valid[b] are zero. */
int b2_get_masks(b2_ctx* ctx, float* masks_host, int64_t capacity_bytes);

/* Stage-addressable access for parity tests.  Activations are returned as fp32. */
int b2_stage_shape(b2_ctx* ctx, const char* name, int64_t shape[4], int32_t* dtype /*0 f32, 1 i32*/);
int b2_get_stage(b2_ctx* ctx, const char* name, void* dst_host, int64_t capacity_bytes);
int b2_set_stage(b2_ctx* ctx, const char* name, const void* src_host, int64_t bytes);
/* Run a subset of the pass: bit mask of B2_PHASE_*. */
enum {
  B2_PHASE_BACKBONE = 1, B2_PHASE_FPN = 2, B2_PHASE_RPN_HEAD = 4, B2_PHASE_PROPOSALS = 8,
  B2_PHASE_ROI = 16, B2_PHASE_HEAD_FC = 32, B2_PHASE_POST = 64, B2_PHASE_BOX_FEAT = 128, B2_PHASE_ALL = 255
};
int b2_run_phases(b2_ctx* ctx, int phase_mask);
/* Device time of the last b2_run_phases/b2_detect per phase (ms), measured with CUDA events. */
int b2_phase_times(b2_ctx* ctx, float ms[8]);
int b2_kernel_launches(b2_ctx* ctx);   /* kernels launched by one full pass */
/* Per-launch-group profiling for the roofline report: device ms of every step of the plan (averaged
 * over `reps` eager passes) and a description of each step (algorithmic FLOPs / HBM bytes). */
int b2_num_steps(b2_ctx* ctx);
int b2_profile_steps(b2_ctx* ctx, int reps, float* ms_out, int cap, int* n_out);
int b2_step_info(b2_ctx* ctx, int idx, char* name, int name_cap, double* flops, double* bytes, int* kind);

/* DeepSORT appearance cost: gallery [S,D] rows grouped per track by seg_offsets[T+1], dets [N,D];
 * cost[T,N] = min over the track's rows of (1 - cos).  Host pointers. */
int b2_cosine_cost(int device, const float* gallery, const int32_t* seg_offsets, int T, const float* dets, int N,
                   int D, int precision, float* cost);

/* ---- DeepSORT association loop in native host code (SURVEY 8f rank 2).  Replaces deep_sort/tracker.py:10-138
 * (Tracker.predict / Tracker.update / _match), track.py:19-166, kalman_filter.py:23-232 (float64 state),
 * linear_assignment.py:12-194 (min_cost_matching, matching_cascade, gate_cost_matrix), iou_matching.py:8-81 and the
 * per-track gallery bookkeeping of nn_matching.py:137-154; scipy.optimize.linear_sum_assignment
 * (linear_assignment.py:5,60) is restated natively with SciPy's tie behaviour.  The appearance cost matrix
 * of every cascade level comes from b2_cosine_cost on `device` (one tensor-core GEMM) unless a cost function is
 * installed (tests install the CPU oracle there; there is no built-in CPU path).
 * b2_tracker_create mirrors Tracker(metric, max_iou_distance, max_age, n_init) + NearestNeighborDistanceMetric("cosine",
 * matching_threshold, budget) (tracker.py:40-48, nn_matching.py:120-131; budget <= 0 = None).
 * b2_tracker_update takes the frame's detections: tlwh [n,4] float64, confidence [n] float64 (may be NULL), features
 * [n,feat_dim] float32 (detection.py:27-42).  b2_tracker_get_tracks copies the live tracks in list order (ids, TrackState
 * 1 tentative / 2 confirmed, hits, age, time_since_update, mean [*,8], covariance [*,64]) and returns their number. */
typedef struct b2_tracker b2_tracker;
typedef int (*b2_appearance_cost_fn)(void* user, const float* gallery, const int32_t* seg_offsets, int T,
                                     const float* dets, int N, int D, float* cost);
int b2_tracker_create(b2_tracker** out, int device, double max_iou_distance, int max_age, int n_init,
                      double matching_threshold, int budget, int feat_dim, int precision);
void b2_tracker_destroy(b2_tracker* trk);
int b2_tracker_set_cost_fn(b2_tracker* trk, b2_appearance_cost_fn fn, void* user);
int b2_tracker_predict(b2_tracker* trk);
int b2_tracker_update(b2_tracker* trk, const double* tlwh, const double* confidence, const float* features, int n);
int b2_tracker_num_tracks(b2_tracker* trk);
int b2_tracker_get_tracks(b2_tracker* trk, int cap, int32_t* ids, int32_t* state, int32_t* hits, int32_t* age,
                          int32_t* time_since_update, double* mean, double* cov);
/* scipy.optimize.linear_sum_assignment on a row-major [nr,nc] float64 matrix: writes min(nr,nc) (row, col) pairs sorted by
 * row, returns their number. */
int b2_linear_sum_assignment(const double* cost, int nr, int nc, int32_t* rows, int32_t* cols);
/* application_util/preprocessing.py:6-74 non_max_suppression(boxes tlwh, max_bbox_overlap, scores): writes the kept
 * indices in pick order, returns their number (scores NULL = order by bottom edge, as the reference). */
int b2_track_nms(const double* tlwh, const double* scores, int n, double max_bbox_overlap, int32_t* keep);

/* ---- TMOT / JDE association in native host code (SURVEY 8f rank 4).  Replaces tmot/matching.py:28-109 and the JDETracker loop
 * of tmot/multitracker.py:13-398 (state float64, embeddings float32).  lap.lapjv (lap 0.4.0) and cython_bbox.bbox_overlaps
 * are third-party and absent from the reference tree: restated from their published algorithms (csrc/tmot.cpp header).
 * b2_lapjv              = lap.lapjv(cost, extend_cost=True, cost_limit) as matching.linear_assignment uses it (:28-38) and
 *                         multi_video_reid.py:512: x[nr] / y[nc] = matched column / row or -1, *opt = matched cost sum.
 * b2_tmot_iou_distance  = matching.iou_distance (:57-77): 1 - IoU(+1 pixel convention) of tlbr boxes, out [na,nb].
 * b2_tmot_fuse_motion   = matching.fuse_motion (:97-109): Kalman gate (chi2inv95 of 4 or 2 dof -> inf) and
 *                         cost = lambda * cost + (1 - lambda) * squared Mahalanobis distance, in place on cost [T,N].
 * b2_tmot_embedding_distance = matching.embedding_distance (:80-94): euclidean distance of track / detection embeddings,
 *                         one tensor-core GEMM on `device` (|a|^2 + |b|^2 - 2ab, then sqrt(max(0, .))), out float64 [T,N]. */
int b2_lapjv(const double* cost, int nr, int nc, double cost_limit, int32_t* x, int32_t* y, double* opt);
int b2_tmot_iou_distance(const double* atlbr, int na, const double* btlbr, int nb, double* out);
int b2_tmot_fuse_motion(const double* means, const double* covs, int T, const double* xyah, int N, double* cost,
                        int only_position, double lambda);
int b2_tmot_embedding_distance(int device, const float* track_feats, int T, const float* det_feats, int N, int D,
                               int precision, double* out);
/* JDETracker(conf_thres, track_max_second_lost, emb_max_dist, iou_max_dist1, iou_max_dist2, emb_smooth_alpha, frame_gap,
 * frame_rate) (multitracker.py:176-204).  Track ids come from a counter shared by every tracker created with the same
 * `share_ids_with` chain (BaseTrack._count is a class attribute, basetrack.py:13,34-37; NULL = own counter).
 * b2_jde_update takes the frame's detections after the pre-tracker NMS: tlwh [n,4] float64, conf [n] float64, features
 * [n,feat_dim] float32 and returns the number of output tracks (tracked and activated, :355).  The embedding distance of
 * the first association comes from b2_distance_matrix on `device` unless a cost function is installed (it then receives
 * one gallery row per track, seg_offsets 0..T, and must write euclidean distances).
 * b2_jde_get_tracks copies list `which` (0 output, 1 tracked_stracks, 2 lost_stracks) in list order; with cap == 0 and
 * ids == NULL it only returns the length. */
typedef struct b2_jde b2_jde;
int b2_jde_create(b2_jde** out, int device, double conf_thres, double track_max_second_lost, double emb_max_dist,
                  double iou_max_dist1, double iou_max_dist2, double emb_smooth_alpha, double frame_gap, double frame_rate,
                  int feat_dim, int precision, b2_jde* share_ids_with);
void b2_jde_destroy(b2_jde* trk);
int b2_jde_set_cost_fn(b2_jde* trk, b2_appearance_cost_fn fn, void* user);
int b2_jde_reset(b2_jde* trk);
/* zeroes only the id counter `trk` shares with its group (multitracker.py:215: reset() of ANY tracker sets BaseTrack._count = 0) */
int b2_jde_reset_ids(b2_jde* trk);
int b2_jde_update(b2_jde* trk, const double* tlwh, const double* conf, const float* features, int n);
int b2_jde_get_tracks(b2_jde* trk, int which, int cap, int32_t* ids, int32_t* state, int32_t* is_activated,
                      int32_t* frame_id, int32_t* start_frame, int32_t* tracklet_len, double* tlwh, double* det_tlwh,
                      double* det_conf, double* score, double* mean, double* cov);

/* ---- ReID embedding: torchreid FeatureExtractor (torchreid/feature_extractor.py:121-252) with osnet_x1_0
 * (torchreid/models/osnet.py:522-534).  b2_reid_create fixes the crop batch; b2_reid_load_weights takes the
 * model's state_dict (torch names, fp32); b2_reid_embed takes host RGB uint8 crops already resized to
 * 256x128 ([n,256,128,3], n <= batch) and returns [n,512] fp32 (ToTensor + Normalize + OSNet eval forward). */
typedef struct b2_reid b2_reid;
int b2_reid_create(b2_reid** out, int device, int batch, int precision);
/* model 0 = osnet_x1_0 as above; model 1 = torchreid's resnet101 (torchreid/models/resnet.py:441-455, the vehicle extractor
 * of single_video_reid.py:410-415): b2_reid_embed then takes crops resized to 128x256 ([n,128,256,3] RGB uint8) and
 * returns [n,2048] (global average pool of layer4, eval mode); state_dict names "conv1.weight", "bn1.*",
 * "layer3.22.conv2.weight", "layer2.0.downsample.0.weight", ... */
int b2_reid_create_model(b2_reid** out, int device, int batch, int precision, int model);
void b2_reid_destroy(b2_reid* ctx);
int b2_reid_load_weights(b2_reid* ctx, const char* const* names, const float* const* data, const int64_t* numel, int n);
int b2_reid_embed(b2_reid* ctx, const uint8_t* crops_host, int n, float* feats_host);
/* Same, with the [n, feat_dim] features left in device memory of the context's GPU (`feats_dev`: e.g. this camera's slice of
 * the gallery buffer the NCCL all-gather of config 5 sends, multi_video_reid.py:448-476) -- a gallery never crosses PCIe. */
int b2_reid_embed_dev(b2_reid* ctx, const uint8_t* crops_host, int n, float* feats_dev);
int b2_reid_feat_dim(b2_reid* ctx);   /* 512 (osnet_x1_0) / 2048 (resnet101) */
int b2_reid_num_launches(b2_reid* ctx);
/* Stage-addressable activation of the last pass as fp32 NHWC (parity tests): "conv1", "maxpool", "conv2.0", ... */
int b2_reid_get_activation(b2_reid* ctx, const char* name, float* dst_host, int64_t capacity_bytes, int64_t shape[4]);

/* ---- EfficientDet (config 3): BiFPN feature network + class/box nets + detection post-processing.
 * Replaces the TF graph of efficientdet/efficientdet_arch.py build_feature_network (:440-505), build_bifpn_layer
 * (:594-682), build_class_and_box_outputs (:343-393) and the wrapper's add_metric_fn_inputs / get_results_tf /
 * own-level ROIAlign box feature (efficientdet_wrapper.py:265-474; anchors.py:399-487). */
typedef struct b2_effdet_config {
  int image_h, image_w;            /* network input size (multiple of 128) */
  int min_level, max_level;        /* 3, 7 */
  int fpn_num_filters, fpn_cell_repeats, box_class_repeats;
  int num_classes, num_scales, num_aspects;
  float aspect_ratios[3][2];       /* (x, y) multipliers, anchors.py:216-257 */
  float anchor_scale;
  int fpn_weight_method;           /* 0 "sum", 1 "fastattn" */
  int backbone_channels[3];        /* channels of the backbone's level 3, 4, 5 endpoints */
  int max_detection_topk;          /* 5000 */
  int result_per_im;               /* 100 */
  float nms_iou_threshold, result_score_thres;
  int precision;                   /* 0 fp16, 1 split (fp32-class) */
  int backbone;                    /* -1: none (b2_effdet_run_features only); 0..7: EfficientNet-b0..b7 trunk
                                    * (efficientdet_arch.py:396-437, backbone/efficientnet_model.py:504-704) */
} b2_effdet_config;
typedef struct b2_effdet b2_effdet;
int b2_effdet_create(b2_effdet** out, const b2_effdet_config* cfg, int device);
void b2_effdet_destroy(b2_effdet* ctx);
/* TF checkpoint variables (names as efficientdet_arch.py creates them, kernels HWIO, fp32) */
int b2_effdet_load_weights(b2_effdet* ctx, const char* const* names, const float* const* data, const int64_t* numel, int n);
/* Backbone endpoints C3/C4/C5 (host NHWC fp32) -> detections: boxes [max][4] x1 y1 x2 y2 scaled by image_scale,
 * scores, classes (1-based), levels, box_feat [max][fpn_num_filters]; *count = number of valid rows. */
int b2_effdet_run_features(b2_effdet* ctx, const float* c3, const float* c4, const float* c5, float image_scale,
                           float* boxes, float* scores, int32_t* classes, int32_t* levels, float* box_feat, int32_t* count);
/* The wrapper's whole per-frame path (efficientdet_wrapper.py:40-111): host BGR uint8 frame [h,w,3] -> build_preprocess
 * (RGB, /255, mean/std, bilinear resize to fit image_h x image_w, zero-pad) -> backbone -> BiFPN -> heads -> detections
 * in frame pixels.  *image_scale_out = image_scale_to_original.  Needs cfg.backbone >= 0. */
int b2_effdet_detect(b2_effdet* ctx, const uint8_t* frame_bgr, int h, int w, float* boxes, float* scores,
                     int32_t* classes, int32_t* levels, float* box_feat, int32_t* count, float* image_scale_out);
/* Stage tensors of the last pass (parity tests): "image", "stem", "block_<i>", "c3".."c5", "fpn3".."fpn7", "cls3".."cls7", "box3".."box7" as fp32 NHWC */
int b2_effdet_get_stage(b2_effdet* ctx, const char* name, float* dst_host, int64_t capacity_bytes, int64_t shape[4]);
int b2_effdet_num_launches(b2_effdet* ctx);
/* Per-step CUDA-event timing / description of the pass (same contract as b2_profile_steps / b2_step_info). */
int b2_effdet_profile_steps(b2_effdet* ctx, int reps, float* ms_out, int cap, int* n_out);
int b2_effdet_step_info(b2_effdet* ctx, int idx, char* name, int name_cap, double* flops, double* bytes, int* kind);

/* Distance matrix of torchreid/distance.py:6-80 on the tensor cores: a [na,D], b [nb,D] (host) -> out [na,nb].
 * metric 0 = cosine (1 - a^.b^), 1 = squared euclidean (|a|^2 + |b|^2 - 2 a.b). */
int b2_distance_matrix(int device, const float* a, int na, const float* b, int nb, int D, int metric, int precision,
                       float* out);

/* ---- Multi-camera ReID track-pair costs (BASELINE config 5; multi_video_reid.py:260-324, 486-512).
 * b2_track_pair_cost = compute_feature_dist (:308-324): crop embeddings of camera 1's tracks a [seg_a[N], D] grouped by
 * seg_a[N+1], camera 2's b / seg_b[M+1] (host, float32); out[i][j] = min over the two tracks' crops of the squared
 * euclidean distance (clamped at 0, as sklearn.euclidean_distances) where gate[i][j] != 0 (gate NULL = all pairs), else
 * `fill` (999 in the reference).  One tensor-core GEMM over the concatenated galleries + one segmented-min kernel.
 * b2_track_spatial_dist = compute_spatial_dist (:260-305) without the ignore-pairs reset: trajectories as (frame, x, y)
 * rows grouped per track, out[i][j] = mean point distance over common frames (camera-2 frames + frame_offset) if <= tol,
 * else 9999.  Host code, float64. */
int b2_track_pair_cost(int device, const float* a, const int32_t* seg_a, int N, const float* b, const int32_t* seg_b,
                       int M, int D, const uint8_t* gate, float fill, int precision, float* out);
/* The same with the galleries already in device memory.  b_dev may be PEER memory of another GPU of the node (opened with
 * b2_gallery_open): the conversion kernel that builds the GEMM's fp16 operand planes then reads the peer gallery over
 * NVLink directly -- the multi-camera exchange without a staged all-gather copy (one process per GPU; each rank scores its
 * share of the camera pairs against the other ranks' galleries in place).
 * b2_gallery_create uploads a gallery [rows, D] into a cudaMalloc'ed buffer and returns the 64-byte CUDA IPC handle other
 * ranks pass to b2_gallery_open (exchange the handles with any host-side channel, e.g. torch.distributed objects);
 * b2_gallery_close unmaps a peer gallery, b2_gallery_free releases an own one (after the peers have closed it).
 * The call runs on a private non-blocking stream and returns when `out` is complete: device inputs must be complete when it
 * is entered (synchronise the stream / collective that produced them first). */
int b2_track_pair_cost_dev(int device, const float* a_dev, const int32_t* seg_a, int N, const float* b_dev,
                           const int32_t* seg_b, int M, int D, const uint8_t* gate, float fill, int precision, float* out);
int b2_gallery_create(int device, const float* feats_host, int rows, int D, float** dev_out, uint8_t handle_out[64]);
int b2_gallery_open(int device, const uint8_t handle[64], float** peer_out);
int b2_gallery_close(int device, float* peer);
int b2_gallery_free(int device, float* dev);
int b2_track_spatial_dist(const int32_t* frames1, const double* pts1, const int32_t* seg1, int N, const int32_t* frames2,
                          const double* pts2, const int32_t* seg2, int M, int frame_offset, double tol, double* out);

/* Single-op entry used by the kernel parity tests (host pointers, NHWC activations, HWIO kernel).  a_mode: -1 automatic,
 * 0 tiled 2-D A operand, 1 im2col; epi_mode: -1 automatic, 0 the direct per-thread epilogue. */
int b2_op_conv2d(int device, const float* x, const float* w, const float* bias, const float* res, int B, int H, int W,
                 int Cin, int R, int S, int Cout, int stride, int dil, int pad_t, int pad_b, int pad_l, int pad_r,
                 int relu, int res_shift, int impl, int split, int a_mode, int epi_mode, float* out);

/* Number of conv launches of this process that ran on CTA pairs (tcgen05 cta_group::2; opt-in through the environment
 * variable B2_PAIR=<min K-blocks>, DESIGN.md 4.3b): lets the tests assert that the hook is live. */
long long b2_conv_pair_launches(void);

#ifdef __cplusplus
}
#endif
#endif  /* B200DET_H_ */
