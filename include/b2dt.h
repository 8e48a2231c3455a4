/* b2dt -- C ABI of the B200-native detect+track hot path.
 *
 * Drop-in boundary (DESIGN.md section 2).  The reference is pure Python and has no FFI; these are
 * the entry points a ctypes binding for its detect+track path needs.  Each entry cites the reference
 * interface it replaces (paths relative to the reference root).  Conventions:
 *   - extern "C", plain pointers and sizes only; every function returns an int status
 *     (B2_OK = 0, negative = error; text via b2_last_error()).
 *   - all tensor memory is caller-owned DEVICE memory unless a parameter says "host";
 *     `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *   - the library owns only its workspaces, activation arena and track banks (opaque handles);
 *     handles are independent: no global mutable state.
 *   - activations are NHWC bf16; "cstride"/"coff" address a channel slice [coff, coff+C) of a
 *     buffer whose pixels are cstride channels apart (this is how torch.cat / chunk disappear).
 */
#ifndef B2DT_H
#define B2DT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_OK 0
#define B2_ERR_ARG (-1)
#define B2_ERR_CUDA (-2)
#define B2_ERR_STATE (-3)
#define B2_ERR_UNSUPPORTED (-4)

#define B2_ACT_NONE 0
#define B2_ACT_SILU 1

const char* b2_last_error(void);
int b2_version(void);
/* number of kernels this library has launched since load (bench.py "gpu_launches") */
long long b2_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Module-level ops (per-layer parity; the engine below is composed of exactly these launches)
 * ---------------------------------------------------------------------------------------------- */

/* Conv.forward_fuse = SiLU(conv2d(x, w', b')) with BN folded, optional fused residual add
 * (ultralytics/nn/modules/conv.py:83-93; Bottleneck.forward block.py:493-495; plain nn.Conv2d 1x1 of
 * Detect head.py:93-96 with act = B2_ACT_NONE).  Implicit GEMM on tcgen05/TMEM, TMA-staged bf16 tiles.
 * in  : [B][H][W][in_cstride] bf16, channels [in_coff, in_coff+Cin)
 * w   : [Cout][k][k][Cin] bf16 (GEMM-K = (kh*k+kw)*Cin + c), bias: [Cout] fp32
 * out : [B][Ho][Wo][out_cstride] bf16, channels [out_coff, out_coff+Cout);  Ho = (H + 2(k/2) - k)/stride + 1
 * residual (may be NULL): same spatial shape as out, added after the activation.
 * Constraints: k in {1,3}; stride in {1,2}; Cin % 16 == 0; cstrides/coffs % 8 == 0. */
int b2_conv2d_bf16(const void* in, int B, int H, int W, int in_cstride, int in_coff, int Cin,
                   const void* w, const float* bias, int Cout, int ksize, int stride, int act,
                   void* out, int out_cstride, int out_coff,
                   const void* residual, int res_cstride, int res_coff, void* stream);

/* Same conv over the channel concatenation [in0 | in1] (Concat, ultralytics/nn/modules/conv.py:673-683, folded into the
 * conv's K loop).  up = 2 marks an input stored at HALF the conv's resolution: nn.Upsample(None, 2, 'nearest')
 * (yolov8-p2.yaml:33,42,47) is folded into the TMA loads (1x1 stride-1 convs only).  H x W: conv input resolution.
 * Weights [Cout][k][k][C0+C1].  in1 may be NULL (single input). */
int b2_conv2d_cat_bf16(const void* in0, int cstride0, int coff0, int C0, int up0,
                       const void* in1, int cstride1, int coff1, int C1, int up1,
                       int B, int H, int W, const void* w, const float* bias, int Cout, int ksize, int stride, int act,
                       void* out, int out_cstride, int out_coff, void* stream);

/* A 3x3 conv (BN folded, SiLU, optional shortcut) and the 1x1 conv that reads its output, as ONE launch: the intermediate tile
 * stays in shared memory as the second GEMM's operand.  Replaces the module pairs Conv -> C2f.cv1 (nn/tasks.py:172-188 with
 * block.py:315-316), Bottleneck.cv2 (+ x) -> C2f.cv2 over cat(y0, y1, m_1..m_n) (block.py:317-319, :493-495; the channels the
 * 1x1 conv reads besides this conv's output are `xC` channels [x_coff, x_coff + xC) of `xsrc`, stored at the conv's OUTPUT
 * resolution, first in the 1x1 conv's K order) and Detect's cv2[l][1] -> cv2[l][2], cv3[l][1] -> cv3[l][2] (head.py:93-100).
 * w: [Cout][3][3][Cin], w2: [Cout2][xC + Cout] bf16; act / act2: B2_ACT_*.  xsrc may be NULL (xC = 0).
 * Returns B2_ERR_UNSUPPORTED when the pair does not fit the chained kernel (b2_conv_chain_plan_ok tells beforehand, without
 * needing a device): run b2_conv2d_bf16 twice then. */
int b2_conv2d_chain_bf16(const void* in, int B, int H, int W, int in_cstride, int in_coff, int Cin,
                         const void* w, const float* bias, int Cout, int ksize, int stride, int act,
                         const void* residual, int res_cstride, int res_coff,
                         const void* xsrc, int x_cstride, int x_coff, int xC,
                         const void* w2, const float* bias2, int Cout2, int act2,
                         void* out, int out_cstride, int out_coff, void* stream);
int b2_conv_chain_plan_ok(int B, int H, int W, int Cin, int Cout, int ksize, int stride, int has_residual, int xC, int Cout2);

/* Stem: letterbox-pad + BGR->RGB + /255 + Conv(3->C0, k3 s2) + SiLU in one pass over uint8 frames, on the tensor
 * cores (data/augment.py:1692-1733 LetterBox pad value 114; engine/predictor.py:152-175 preprocess; model.0 of
 * yolov8-p2.yaml).  frames: [B][src_h][src_w][3] uint8 BGR.  The letterboxed canvas is H x W with the frame at
 * (pad_top, pad_left).  w: [C0][32] bf16, BN-folded, GEMM-K index (kh*3+kw)*3 + c_rgb, entries 27..31 zero, NOT
 * divided by 255 (the epilogue scales in fp32).  bias: [C0] fp32.  out: [B][H/2][W/2][out_cstride] bf16. */
int b2_stem_u8(const uint8_t* frames, int B, int src_h, int src_w, int H, int W, int pad_top, int pad_left,
               const void* w, const float* bias, int C0, void* out, int out_cstride, int out_coff, void* stream);
/* Same stem for float tensors BCHW RGB in [0,1] (data/loaders.py:566-638 LoadTensor): the tensor core consumes
 * bf16(255 x), exact for uint8-derived inputs.  dtype: 0 fp32, 1 bf16 */
int b2_stem_f32(const void* bchw, int dtype, int B, int H, int W, const void* w, const float* bias, int C0,
                void* out, int out_cstride, int out_coff, void* stream);

/* Stand-alone preprocess (engine/predictor.py:152-175 + LetterBox pad-only path): uint8 HWC BGR ->
 * fp32 BCHW RGB in [0,1], canvas H x W, border 114/255.  For API parity (BasePredictor.preprocess). */
int b2_preprocess_u8(const uint8_t* frames, int B, int src_h, int src_w, int H, int W, int pad_top, int pad_left,
                     float* out_bchw, void* stream);
/* cv2.resize(INTER_LINEAR) on uint8 HWC (data/augment.py:1718): fixed-point bilinear identical to OpenCV. */
int b2_resize_bilinear_u8(const uint8_t* src, int B, int sh, int sw, uint8_t* dst, int dh, int dw, void* stream);
/* LetterBox (data/augment.py:1692-1733) for a ragged batch: image b is src_h x src_w HWC BGR at byte offset src_off[b] of `src`
 * (16-byte aligned offsets take the vector copy path); it is resized to rh x rw with the arithmetic of b2_resize_bilinear_u8
 * (copied when the shape is unchanged) and placed at (top, left) of canvas b; everything else is 114.
 * src_off: device int64 [B]; geom: device int32 [B][6] {src_h, src_w, rh, rw, top, left}; canvas: [B][H][W][3] uint8,
 * W a multiple of 16, at most 4096.  A placement that does not fit the canvas leaves that canvas at 114. */
int b2_letterbox_u8(const uint8_t* src, const int64_t* src_off, const int32_t* geom, int B, int H, int W, uint8_t* canvas, void* stream);

/* SPPF pooling (block.py:237-241): y1 = maxpool5(x), y2 = maxpool5(y1), y3 = maxpool5(y2) (stride 1, pad 2).
 * buf: [B][H][W][cstride] bf16; reads channels [coff, coff+C), writes [coff+C, coff+4C). */
int b2_sppf_pool(void* buf, int B, int H, int W, int cstride, int coff, int C, void* stream);

/* nn.Upsample(None, 2, 'nearest') / channel-slice copy written into a concat slice
 * (yolov8-p2.yaml:33-54, conv.py:673-683 Concat).  scale in {1,2}. */
int b2_upsample_slice(const void* in, int B, int H, int W, int in_cstride, int in_coff, int C, int scale,
                      void* out, int out_cstride, int out_coff, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Detect post-processing
 * ---------------------------------------------------------------------------------------------- */

/* Detect._inference + confidence filter (head.py:152-187, block.py:78-81 DFL, tal.py:367-391,
 * nms.py:74 `amax > conf`, :111 best class): reads per-level NHWC bf16 logits
 * [B][h_l*w_l][lstride] (64 DFL bins then nc class logits) and appends one candidate per anchor whose
 * best class score > conf:  cand[b][i] = {x1,y1,x2,y2 (letterboxed-input pixels), score, cls} fp32,
 * cand_idx[b][i] = anchor index, cand_count[b].  At most cand_cap candidates per image are stored
 * (count keeps counting).  classes_mask: optional nc uint8 (nms.py:120-124 `classes=` filter).
 * dense_out (may be NULL): the reference-shaped (B, 4+nc, A) fp32 tensor [cx,cy,w,h,sigmoid(cls)...]. */
int b2_decode(const void* const* level_logits, const int* level_h, const int* level_w, const int* level_stride,
              int n_levels, int B, int nc, int lstride, float conf, const uint8_t* classes_mask,
              float* cand, int32_t* cand_idx, int32_t* cand_count, int cand_cap, float* dense_out, void* stream);

/* Candidate stage fed by the FUSED Detect head (b2_engine_head): per level, dist [B][h*w][4] fp32 (DFL expectations
 * l,t,r,b in grid units) and cls [B][h*w][2] fp32 {best class logit, class}; the DFL softmax / class max run in the
 * epilogue of the head's last convs, so the (64+nc)-channel logits are never written.  Same outputs as b2_decode. */
int b2_candidates_from_head(const float* const* level_dist, const float* const* level_cls, const int* level_h, const int* level_w,
                            const int* level_stride, int n_levels, int B, float conf, const uint8_t* classes_mask,
                            float* cand, int32_t* cand_idx, int32_t* cand_count, int cand_cap, void* stream);

/* Candidate stage of non_max_suppression for callers that hold the reference-shaped dense tensor
 * pred (B, no = 4+nc(+extra), A) fp32 [cx,cy,w,h,scores...] (utils/nms.py:74 `amax > conf`, :85-87 xywh2xyxy,
 * :111-113 best class, :120-124 classes filter).  Same candidate layout as b2_decode. */
int b2_candidates_from_dense(const float* pred, int B, int nc, int no, int A, float conf, const uint8_t* classes_mask,
                             float* cand, int32_t* cand_idx, int32_t* cand_count, int cand_cap, void* stream);

/* non_max_suppression tail + scale_boxes/clip_boxes (utils/nms.py:129-160; torchvision.ops.nms or
 * TorchNMS.nms :237-304; utils/ops.py:105-138,157-183).  Per image: sort candidates by (score desc,
 * anchor asc), cap at max_nms, greedy NMS on class-offset fp32 boxes (cls*max_wh unless agnostic),
 * suppress iou > iou_thres, keep <= max_det, then subtract (pad_x,pad_y), divide by gain, clip to
 * (orig_w, orig_h).  mode: 0 = exact greedy (torchvision branch), 1 = legacy TorchNMS early exit.
 * out: [B][max_det][6] {x1,y1,x2,y2,conf,cls}; out_count[B]; out_idx (may be NULL): kept anchor ids. */
int b2_nms(const float* cand, const int32_t* cand_idx, const int32_t* cand_count, int cand_cap, int B,
           float iou_thres, int max_det, int max_nms, int agnostic, float max_wh, int mode,
           float gain, float pad_x, float pad_y, float orig_w, float orig_h, int do_scale,
           float* out, int32_t* out_count, int32_t* out_idx, void* workspace, size_t workspace_bytes, void* stream);
/* b2_nms with scale_boxes + clip_boxes per image: scale is a device float [B][5] {gain, pad_x, pad_y, orig_w, orig_h}, row b
 * applied to image b with the same operations as the scalar epilogue (a batch of frames of different original shapes). */
int b2_nms_scaled(const float* cand, const int32_t* cand_idx, const int32_t* cand_count, int cand_cap, int B,
                  float iou_thres, int max_det, int max_nms, int agnostic, float max_wh, int mode, const float* scale,
                  float* out, int32_t* out_count, int32_t* out_idx, void* workspace, size_t workspace_bytes, void* stream);
size_t b2_nms_workspace_bytes(int B, int cand_cap);

/* ------------------------------------------------------------------------------------------------
 * Engine: the whole YOLOv8-P2 forward as one launch plan (nn/tasks.py:159-188 _predict_once over
 * the fused graph; replaces AutoBackend.forward nn/autobackend.py:608-637 for the pt branch).
 * `plan` is the int32 program emitted by the host (engine.py); `weights` a host blob it indexes.
 * ---------------------------------------------------------------------------------------------- */
typedef struct b2_engine b2_engine_t;
int b2_engine_create(const int32_t* plan, int plan_words, const void* weights_host, size_t weight_bytes,
                     int B, int H, int W, b2_engine_t** out);
int b2_engine_destroy(b2_engine_t* e);
/* frames: [B][src_h][src_w][3] uint8 BGR device memory, placed at (pad_top,pad_left) of the HxW canvas */
int b2_engine_forward_u8(b2_engine_t* e, const uint8_t* frames, int src_h, int src_w, int pad_top, int pad_left, void* stream);
/* Same forward, launched eagerly with a CUDA event between consecutive launches; fills the device time of each
 * launch (ms_per_op: host, [b2_engine_num_launches]; op 0 = stem).  Synchronises.  For roofline accounting. */
int b2_engine_profile_u8(b2_engine_t* e, const uint8_t* frames, int src_h, int src_w, int pad_top, int pad_left,
                         float* ms_per_op, void* stream);
/* x: BCHW RGB [0,1], dtype 0 fp32 / 1 bf16 */
int b2_engine_forward_f32(b2_engine_t* e, const void* bchw, int dtype, void* stream);
/* Per-level head logits of the last forward: device pointers, [B][h*w][lstride] bf16 */
int b2_engine_levels(b2_engine_t* e, int* n_levels, const void** logits, int* h, int* w, int* stride, int* lstride);
/* Fused Detect head outputs of the last forward (engines lowered with the fused head): per level device pointers
 * dist [B][h*w][4] fp32, cls [B][h*w][2] fp32.  B2_ERR_STATE if the engine writes plain logits instead. */
int b2_engine_head(b2_engine_t* e, const float** dist, const float** cls);
/* Debug/parity: device pointer + geometry of activation buffer `buf` (NHWC bf16) */
int b2_engine_buffer(b2_engine_t* e, int buf, const void** ptr, int* h, int* w, int* c);
size_t b2_engine_arena_bytes(b2_engine_t* e);
int b2_engine_num_launches(b2_engine_t* e);
/* 1 = replay the layer launches from a captured CUDA graph (default), 0 = eager launches */
int b2_engine_use_graph(b2_engine_t* e, int on);

/* ------------------------------------------------------------------------------------------------
 * Tracker: structure-of-arrays Kalman bank, one independent tracker per stream
 * (kalman/enhanced_multi_target_tracker.py:15-132 EnhancedMultiTargetTracker.update,
 *  kalman/enhanced_aircraft_kalman_tracker.py:23-405 AircraftKalmanTracker).
 * ---------------------------------------------------------------------------------------------- */
#define B2_TRACK_COLS 20
/* output row (fp32 unless noted; "i32" columns are int32 bit patterns):
 *  0 id(i32) 1..4 bbox x1,y1,x2,y2 5 confidence 6 predicted(i32: 1 = 'predicted', 0 = 'detected')
 *  7 age(i32) 8 hits(i32) 9 hit_streak(i32) 10 time_since_update(i32) 11 lost_frames(i32, = tsu)
 *  12 is_lost(i32) 13 vx 14 vy 15 motion_confidence 16 is_stable_motion(i32) 17 speed 18 direction 19 slot(i32) */
#define B2_TRAJ_LEN 30
typedef struct b2_tracker b2_tracker_t;
int b2_tracker_create(int n_streams, int capacity, int max_dets, int max_lost_frames, int min_hits,
                      float iou_threshold, b2_tracker_t** out);
/* mode 1: the same bank driven by the rules of camera_motion_compensation/motion_compensated_multi_tracker.py:75-283 (update
 * without a frame) over MotionResetKalmanTracker tracks (motion_reset_kalman_tracker.py:16-355): per-track position-jump /
 * velocity-change / size-change detectors with a 15-frame cooldown, reset = state overwritten by the detection with the
 * covariance rescaled, the association box blended towards the last stored position for 10 frames after a reset, candidates
 * IoU > threshold with ties to the LARGER (detection, track), every live track reported.  stats (b2_tracker_export /
 * b2_tracker_stats): slots 3 / 4 hold individual_resets / tracking_recoveries ([6], [7] of b2_tracker_stats). */
int b2_tracker_create_ex(int n_streams, int capacity, int max_dets, int max_lost_frames, int min_hits,
                         float iou_threshold, int mode, b2_tracker_t** out);
int b2_tracker_destroy(b2_tracker_t* t);
int b2_tracker_reset(b2_tracker_t* t, void* stream);
/* b2_tracker_reset for the streams with flags_dev[s] != 0 ([n_streams] int32, device): their slots, counters, frame count and
 * mode-1 fields are cleared and next_id set to 1; other streams are not touched.  Ordered on `stream`, no host synchronisation. */
int b2_tracker_reset_streams(b2_tracker_t* t, const int32_t* flags_dev, void* stream);
/* The reference's track list is unbounded (enhanced_multi_target_tracker.py:92-101 appends); the bank is not.  A caller that
 * sees `active + max_dets > capacity` (b2_tracker_stats / b2_tracker_export) enlarges the bank in place: every slot keeps its
 * index, state and id.  Synchronises `stream`.  Output buffers of b2_tracker_update must be re-sized by the caller. */
int b2_tracker_capacity(b2_tracker_t* t);
int b2_tracker_grow(b2_tracker_t* t, int new_capacity, void* stream);
/* Device-side snapshot of the per-stream counters, [n_streams][8] int64 {created, terminated, active, long_term_predictions,
 * recoveries, dropped (detections that found no free slot; the reference never drops), 0, 0}, ordered on `stream`:
 * a pipeline downloads it with its rows instead of synchronising on b2_tracker_export. */
int b2_tracker_stats(b2_tracker_t* t, long long* stats_dev_out, void* stream);
/* One frame for every stream.  dets: [n_streams][max_dets][det_cols] fp32 rows starting with
 * x1,y1,x2,y2 (det_cols >= 4, e.g. 6 for NMS output rows); det_counts: [n_streams] int32.  All max_dets rows of a stream must be
 * allocated: rows past the count are requested before the count is known and ignored (their contents do not matter).
 * out_rows: [n_streams][out_cap][B2_TRACK_COLS]; out_counts: [n_streams] int32 = tracks reported (rows beyond out_cap are
 * counted but not written: out_counts[s] > out_cap tells the caller its buffer was too small);
 * out_traj (may be NULL): [n_streams][out_cap][B2_TRAJ_LEN][2] fp32 last centres, oldest first,
 * out_traj_len (NULL iff out_traj is): [n_streams][out_cap] int32.
 * Row order per stream is deterministic but not by id (tracks no detection overlaps first, slot order; then the tracks with a
 * candidate detection; then new tracks): order by column 0 for the reference's list order. */
int b2_tracker_update(b2_tracker_t* t, const float* dets, int det_cols, const int32_t* det_counts,
                      float* out_rows, int32_t* out_counts, float* out_traj, int32_t* out_traj_len, int out_cap, void* stream);
/* The same with the per-row extras of a mode-1 bank: out_extra (may be NULL): [n_streams][out_cap][4]
 * {reset_count (i32), frames_since_reset (i32), motion_consistency (fp32), 0} (get_track_info, motion_reset_kalman_tracker.py:323-342). */
int b2_tracker_update_ex(b2_tracker_t* t, const float* dets, int det_cols, const int32_t* det_counts,
                         float* out_rows, int32_t* out_counts, float* out_traj, int32_t* out_traj_len, float* out_extra,
                         int out_cap, void* stream);
/* mode-1 bank, one stream (synchronises): reset_host [cap][8] {id, reset_count, last_reset_frame, (i32 bits) motion_consistency (fp32),
 * len(position_history), len(motion_scores), len(bbox_history) (i32 bits), 0}, slot order. */
int b2_tracker_export_reset(b2_tracker_t* t, int stream_idx, float* reset_host, int32_t* n_tracks_host);
/* Host-side inspection (synchronises): dense state of one stream.  x: [cap][8], P: [cap][64] (dense 8x8
 * rebuilt from the decoupled blocks), meta: [cap][8] int32 {id, age, hits, hit_streak, tsu, lost_frames, is_lost, n_vel},
 * stats: [8] int64 {created, terminated, active, long_term_predictions, recoveries, frame_count, next_track_id,
 * dropped (detections that found no free slot)}.  Any of the host pointers may be NULL. */
int b2_tracker_export(b2_tracker_t* t, int stream_idx, float* x_host, float* P_host, int32_t* meta_host,
                      int32_t* n_tracks_host, long long* stats_host);
/* Motion analysis of one stream's live tracks (analyze_motion_pattern, enhanced_aircraft_kalman_tracker.py:137-163; read by
 * get_statistics :288-304): motion_host [cap][8] fp32 {id (i32 bits), velocity_avg x, y, direction, speed, stability_score,
 * prediction_confidence, n_velocities (i32 bits)}, slot order.  Synchronises. */
int b2_tracker_export_motion(b2_tracker_t* t, int stream_idx, float* motion_host, int32_t* n_tracks_host);
/* bytes of bank state + output row read and written per track and frame (roofline accounting): `predict_bytes` for a
 * coasting track (finished by the sweep: predict, mark lost, delete test, row), `update_bytes` for a matched one */
int b2_tracker_bytes_per_track(int* predict_bytes, int* update_bytes);
/* AircraftKalmanTracker.predict (enhanced_aircraft_kalman_tracker.py:184-203) alone on every live track of the bank */
int b2_tracker_bank_predict(b2_tracker_t* t, void* stream);
int b2_tracker_seed(b2_tracker_t* t, const float* boxes, const int32_t* counts, int max_rows, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Ultralytics ByteTrack/BoT-SORT Kalman filters (ultralytics/trackers/utils/kalman_filter.py:
 * KalmanFilterXYAH :39-286, KalmanFilterXYWH :289-493), batched over N tracks, dense 8x8 fp32.
 * kind: 0 = XYAH, 1 = XYWH.  mean [N][8], cov [N][64] row-major, measurements [.][4].
 * ---------------------------------------------------------------------------------------------- */
int b2_kf_initiate(int kind, const float* meas, float* mean, float* cov, int N, void* stream);
int b2_kf_predict(int kind, float* mean, float* cov, int N, void* stream);           /* multi_predict, in place */
int b2_kf_project(int kind, const float* mean, const float* cov, float* pmean, float* pcov, int N, void* stream);
int b2_kf_update(int kind, float* mean, float* cov, const float* meas, const uint8_t* mask, int N, void* stream);
/* out[n][m] = gating distance of track n to measurement m; metric 0 = 'maha', 1 = 'gaussian' */
int b2_kf_gating(int kind, const float* mean, const float* cov, int N, const float* meas, int M,
                 int only_position, int metric, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Association of the upstream tracker plug-in (ByteTrack / BoT-SORT), batched over S independent problems (one per video
 * stream and association stage).  Problem s has na[s] <= n_max rows (tracks) and nb[s] <= m_max columns (detections);
 * na / nb NULL: every problem is n_max x m_max.  boxes: [S][n_max][4] / [S][m_max][4] xyxy fp32 (16-byte aligned),
 * cost: [S][n_max][m_max] fp32 (entries outside a problem's na x nb corner are not touched).
 * ---------------------------------------------------------------------------------------------- */
/* matching.iou_distance (ultralytics/trackers/utils/matching.py:66-113: 1 - bbox_ioa(a, b, iou=True), utils/metrics.py:19-52)
 * and, when scores_b [S][m_max] is given, matching.fuse_score (:135-157): 1 - (1 - cost) * score -- float32, reference op order */
int b2_iou_cost(const float* boxes_a, const float* boxes_b, const float* scores_b, const int32_t* na, const int32_t* nb,
                int S, int n_max, int m_max, float* cost, void* stream);
/* matching.linear_assignment(cost, thresh) on its default branch (matching.py:20-63: lap.lapjv(cost, extend_cost=True,
 * cost_limit=thresh)): x_out [S][n_max] = matched column of each row or -1, y_out [S][m_max] = matched row of each column or -1.
 * Exact optimum (float64 shortest augmenting paths), one CTA per problem. */
int b2_linear_assignment(const float* cost, const int32_t* na, const int32_t* nb, int S, int n_max, int m_max, float thresh,
                         int32_t* x_out, int32_t* y_out, void* stream);
/* The same solver on a float64 cost [S][n_max][m_max] with a float64 threshold (lap.lapjv works in double: the BoT-SORT ReID cost
 * is float64 and can hold entries closer to the threshold than float32 resolves). */
int b2_linear_assignment_f64(const double* cost, const int32_t* na, const int32_t* nb, int S, int n_max, int m_max, double thresh,
                             int32_t* x_out, int32_t* y_out, void* stream);
/* BOTSORT.get_dists with ReID (ultralytics/trackers/bot_sort.py:154-232, matching.embedding_distance):
 *   d    = iou_distance (float32, as b2_iou_cost);  mask = d > prox_limit (float32; prox_limit = float32(1 - proximity_thresh))
 *   d    = fuse_score(d) when scores_b is given (float32)
 *   emb  = max(0, cdist(feat_a, feat_b, 'cosine')) / 2 in float64;  emb[emb > app_limit] = 1 (app_limit = 1 - appearance_thresh);
 *   emb[mask] = 1;  cost = minimum(d, emb) float64 [S][n_max][m_max] (entries outside a problem's corner are not touched).
 * feat_a: track smooth features [S][n_max][D], feat_b: detection features [S][m_max][D], fp32. */
int b2_botsort_cost(const float* boxes_a, const float* boxes_b, const float* scores_b, const int32_t* na, const int32_t* nb,
                    const float* feat_a, const float* feat_b, int D, int S, int n_max, int m_max, float prox_limit, double app_limit,
                    double* cost, void* stream);

/* ------------------------------------------------------------------------------------------------
 * BoT-SORT ReID on the detector's own features (botsort.yaml with_reid: True, model: auto)
 * ---------------------------------------------------------------------------------------------- */
/* get_obj_feats (models/yolo/detect/predict.py): out[b][k][0..s) = row of kept detection k of image b in the Detect input map of its
 * level, averaged over groups of C_l / s consecutive channels (fp32, not normalised).  Level l (host arrays, Detect order): NHWC
 * bf16 buffer level_ptr[l] [B][h][w][cstride], channels [coff, coff + C); anchor ids count the levels' h*w pixels in that order.
 * det_idx [B][max_det] (b2_nms out_idx), det_count [B].  Every C_l must be a multiple of s.  Rows k >= det_count[b] are not written. */
int b2_reid_gather(const void* const* level_ptr, const int* level_h, const int* level_w, const int* level_cstride, const int* level_coff,
                   const int* level_c, int n_levels, const int32_t* det_idx, const int32_t* det_count, int B, int max_det, int s,
                   float* out, void* stream);
/* BOTrack.update_features (bot_sort.py) for N rows, float32: curr [N][D] /= |curr| in place; where has_smooth[r] (NULL: no row)
 * smooth = 0.9 smooth + 0.1 curr, otherwise smooth = curr; then smooth /= |smooth| (a first smooth is the same vector as curr in
 * the reference, so curr receives that renormalisation too). */
int b2_reid_update(float* curr, float* smooth, const uint8_t* has_smooth, int N, int D, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Global camera motion (camera_motion_compensation/global_motion_detector.py, method 'optical_flow', and the global-reset rule of
 * motion_compensated_multi_tracker.py:75-146), batched over S streams.  Frames are HWC BGR uint8 at per-stream byte offsets
 * (frame_off_dev, int64 [S], the layout of b2_letterbox_u8).  Only the reference's parameters are supported; others return
 * B2_ERR_UNSUPPORTED.  Frames of any size: LK starts, per stream, at the deepest level larger than the 21x21 window (cv2's rule).
 * ---------------------------------------------------------------------------------------------- */
/* Host-only layout of a gray pyramid buffer (4 levels per stream, back to back): shapes_host [S][2] {h, w};
 * level_off_host [S][4] byte offsets, level_hw_host [S][4][2], pix_off_host [S] offsets of level 0 in pixels (the response buffer
 * of b2_corner_min_eig), totals_host [2] {pyramid bytes, level-0 pixels}. */
int b2_pyramid_layout(int n_streams, const int* shapes_host, long long* level_off_host, int* level_hw_host, long long* pix_off_host,
                      long long* totals_host);
/* cv2.cvtColor(BGR2GRAY) and three cv2.pyrDown levels, bit-exact.  max_h / max_w: the largest frame. */
int b2_gray_pyramid_u8(const uint8_t* frames, const long long* frame_off_dev, int n_streams, int max_h, int max_w,
                       uint8_t* pyr, const long long* level_off_dev, const int* level_hw_dev, void* stream);
/* cv2.cornerMinEigenVal(level 0, blockSize=7, ksize=3) -> eig_out fp32 at pix_off (within 1e-5 of the maximum of cv2's). */
int b2_corner_min_eig(const uint8_t* pyr, const long long* level_off_dev, const int* level_hw_dev, const long long* pix_off_dev,
                      int n_streams, int max_h, int max_w, int block_size, int ksize, float* eig_out, void* stream);
/* goodFeaturesToTrack's selection (maxCorners=200, qualityLevel=0.01, minDistance=15) on a response: local 3x3 maxima above
 * 0.01 max off the one-pixel border, ordered by value then linear index (both descending), accepted greedily at squared distance
 * >= 225.  corners_out [S][200][2] fp32 (x, y), counts_out [S].  workspace: b2_good_features_workspace_bytes(S, total_pixels). */
size_t b2_good_features_workspace_bytes(int n_streams, long long total_pixels);
int b2_good_features(const float* eig, const long long* pix_off_dev, const int* level_hw_dev, int n_streams, int max_h, int max_w,
                     long long total_pixels, int max_corners, double quality_level, double min_distance, void* workspace,
                     size_t workspace_bytes, float* corners_out, int* counts_out, void* stream);
/* cv2.calcOpticalFlowPyrLK(winSize=21x21, maxLevel=3, criteria COUNT|EPS 30 / 0.01) between two pyramids of the same layout:
 * pts [S][max_pts][2], counts [S]; next_out [S][max_pts][2], status_out [S][max_pts] uint8 (rows past a count are not written). */
int b2_lk_pyr(const uint8_t* prev_pyr, const uint8_t* next_pyr, const long long* level_off_dev, const int* level_hw_dev, int n_streams,
              const float* pts, const int* counts, int max_pts, int win, int max_level, int max_count, double epsilon,
              float* next_out, uint8_t* status_out, void* stream);

/* The per-stream detector and its decision state on the device.  b2_motion_flow: pyramid of the frame (the previous frame's is
 * kept), then corners of the previous frame and their flow into this one -- needs the frames only.  b2_motion_decide (once per
 * flow): detect_motion's vector / thresholds and _should_global_reset from det_counts_dev [S] (this frame's detections, NULL = 0);
 * flags_dev [S] int32 = 1 where every track of the stream is to be dropped (feed b2_tracker_reset_streams); info_dev [S][8] fp32
 * {magnitude, vx, vy, is_motion, should_reset, global_reset, corners, tracked}.  tracker_stats_dev (b2_tracker_stats of the bank
 * before the reset, may be NULL) feeds the individual-resets / recoveries base.  b2_motion_stats: [S][8] float64 {total_detections,
 * motion_events, reset_triggers, avg_motion_magnitude, global_motion_events, global_resets, base individual_resets,
 * base tracking_recoveries}. */
typedef struct b2_motion b2_motion_t;
int b2_motion_create(int n_streams, const int* shapes_host, b2_motion_t** out);
int b2_motion_flow(b2_motion_t* m, const uint8_t* frames, const long long* frame_off_dev, void* stream);
int b2_motion_decide(b2_motion_t* m, const int32_t* det_counts_dev, const long long* tracker_stats_dev, int32_t* flags_dev,
                     float* info_dev, void* stream);
int b2_motion_stats(b2_motion_t* m, double* stats_dev_out, void* stream);
int b2_motion_reset(b2_motion_t* m, void* stream);
int b2_motion_destroy(b2_motion_t* m);

#ifdef __cplusplus
}
#endif
#endif /* B2DT_H */
