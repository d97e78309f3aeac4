/* dvfe.h — C ABI of the B200-native Dynamic-VINS feature-tracking front-end.
 *
 * This is the drop-in boundary for the hot path named in BASELINE.json `north_star`.
 * The reference has no FFI layer: the seam is a C++ class API inside one binary
 * (SURVEY.md §8b).  Every entry point below names the reference interface it
 * replaces (paths under /root/reference/dynamic_vins/src/).  Plain pointers and
 * sizes only; no C++/torch types cross this boundary; nothing throws — the
 * reference's exception cases come back as negative codes.
 *
 * One `dvfe_tracker` owns B independent camera streams of identical geometry on
 * one GPU ("stream-sharded replicas", SURVEY.md §8e).  B = 1 is the reference's
 * single `FeatureTracker` + `InstsFeatManager` pair.  All device state (pyramids,
 * point sets, ids, velocities) stays resident in HBM between calls.
 */
#ifndef DVFE_H_
#define DVFE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVFE_OK 0
#define DVFE_ERR_INVALID (-1)   /* bad argument / empty input: std::runtime_error, front_end/feature_utils.cpp:39-41 */
#define DVFE_ERR_CUDA (-2)      /* CUDA runtime failure (see dvfe_last_error) */
#define DVFE_ERR_CONFIG (-3)    /* bad settings path or key: front_end/front_end_parameters.cpp:20-22 */
#define DVFE_ERR_CAPACITY (-4)  /* a caller-provided buffer or a configured capacity is too small */
#define DVFE_ERR_NO_DEVICE (-5) /* no sm_100 device: the library has no CPU fallback */

#define DVFE_MAX_PYR_LEVELS 5

/* camodocal PinholeCamera parameters (model_type: PINHOLE — the only model any shipped config uses;
 * /root/reference/camera_models/src/camera_models/PinholeCamera.cc:187-205) */
typedef struct dvfe_camera {
    double fx, fy, cx, cy;
    double k1, k2, p1, p2;
} dvfe_camera;

/* fe_para / cfg keys the path reads (front_end/front_end_parameters.cpp:24-37, utils/parameters.cpp) */
typedef struct dvfe_config {
    int width, height;          /* image_width, image_height */
    int n_streams;              /* B independent streams held by this tracker (reference: 1) */
    int stereo;                 /* cfg::is_stereo (num_of_cam == 2) */
    int max_cnt;                /* max_cnt */
    int min_dist;               /* min_dist */
    int max_dynamic_cnt;        /* max_dynamic_cnt */
    int min_dynamic_dist;       /* min_dynamic_dist */
    int flow_back;              /* flow_back (fe_para::is_flow_back) */
    int use_mask_morphology;    /* use_mask_morphology */
    int mask_morphology_size;   /* mask_morphology_size */
    int lk_max_level;           /* 3: cv::calcOpticalFlowPyrLK(..., Size(21,21), 3), front_end/feature_utils.cpp:43 */
    int max_instances;          /* per-stream instance slots for dynamic mode (0 = raw mode only) */
    int device;                 /* CUDA device ordinal */
    dvfe_camera cam0, cam1;     /* cam_t.cam0 / cam_t.cam1, utils/camera_model.h:52-54 */
    int n_groups;               /* 0/1: one launch set for all streams.  G > 1: the streams are split into G groups that
                                 * run on their own CUDA streams, so the latency-bound phases of one group (corner
                                 * selection, small kernels, launch tails) overlap the throughput-bound kernels of the
                                 * others (+10..13 % frames/s at 64 streams); results are identical */
    int reserved;
} dvfe_config;

/* One observation of FeatureBackground::points — map<id, vector<pair<cam, Vec7d>>>
 * (basic/frontend_feature.h:34-47; packed by FeatureTracker::SetOutputFeats,
 * front_end/background_tracker.cpp:340-392).  v = [x, y, 1, u, v, vx, vy]. Records come
 * sorted by (id, cam), i.e. in the iteration order of the reference's std::map. */
typedef struct dvfe_obs {
    uint32_t id;
    int32_t cam;
    double v[7];
} dvfe_obs;

/* One feature of FeatureInstance::features (basic/frontend_feature.h:49-58, basic/point_feature.h:22-100;
 * packed by InstsFeatManager::Output, front_end/dynamic_tracker.cpp:521-577). */
typedef struct dvfe_inst_obs {
    uint32_t inst_id;           /* instance (track) id */
    uint32_t id;                /* feature id */
    int32_t is_stereo;
    int32_t reserved;
    double point[3];            /* (un.x, un.y, 1) */
    double vel[2];
    double point_right[3];
    double vel_right[2];
    double uv[2];               /* ROI-local pixel position (curr_points) */
    double disp;                /* prev_img.disp.at<float>(curr_points[i]): the caller's map read at the ROI-LOCAL position
                                 * (front_end/dynamic_tracker.cpp:547, reference quirk Q8); 0 when dvfe_inst_in::disp is NULL */
} dvfe_inst_obs;

/* One detected instance of a frame: Box2D + InstRoi (basic/box2d.h:24-56), as produced by
 * SemanticImage::SetMaskAndRoi (basic/semantic_image.cpp:20-63) and consumed by
 * InstsFeatManager::AddViodeInstances (front_end/dynamic_tracker.cpp:585-605). */
typedef struct dvfe_inst_in {
    uint32_t track_id;
    int32_t x, y, w, h;         /* Box2D::rect (integer valued) */
    const uint8_t* mask;        /* HOST pointer, h rows x w cols, 255 = object (InstRoi::mask_cv) */
    int32_t mask_pitch;
    const float* disp;          /* HOST pointer to SemanticImage::disp of this frame (CV_32F, full image size, the same for
                                 * every box of the stream) or NULL; must stay valid until the step's records are read
                                 * (dvfe_insts_track returns / dvfe_wait) */
    int32_t disp_pitch;         /* bytes per row of disp */
    int32_t label_bit;          /* with DVFE_DYN_LABELS: the bit of the frame's label image that marks this instance's pixels
                                 * (`mask` is then ignored and may be NULL); otherwise unused */
} dvfe_inst_in;

typedef struct dvfe_tracker dvfe_tracker;

/* ---- lifetime --------------------------------------------------------------------- */

/* FeatureTracker::FeatureTracker(config_path) + InstsFeatManager::InstsFeatManager(config_path)
 * (front_end/background_tracker.cpp:30-43, front_end/dynamic_tracker.cpp:33) with the yaml already parsed. */
int dvfe_create(const dvfe_config* cfg, dvfe_tracker** out);
void dvfe_destroy(dvfe_tracker* t);

/* fe_para::SetParameters(config_path) + the cfg keys of utils/parameters.cpp + the two camodocal yaml files
 * named by cam0_calib / cam1_calib (front_end/front_end_parameters.cpp:17-40).  Fills *cfg; n_streams = 1. */
int dvfe_config_from_yaml(const char* config_path, dvfe_config* cfg);

const char* dvfe_last_error(const dvfe_tracker* t);   /* t may be NULL: last error of dvfe_create / ops */
const char* dvfe_version(void);
/* Number of CUDA kernels this library has launched in this process (bench.py `gpu_launches`). */
unsigned long long dvfe_kernel_launches(void);

/* Run this tracker's work on a caller-owned CUDA stream (a cudaStream_t passed as void*), so the caller can
 * bracket steps with its own events.  Default: a private non-blocking stream. */
int dvfe_set_stream(dvfe_tracker* t, void* cuda_stream);

/* Per-stage device timers (CUDA events on the tracker's stream around each stage of the frame step; the
 * reference logs the same split with TicToc, front_end/background_tracker.cpp:72,98,105,138).
 * dvfe_profile(t, 1) resets and enables, dvfe_profile(t, 0) disables.  dvfe_profile_read returns the number of
 * stages; names[i] / total_ms[i] (caller arrays of >= 16 entries) get the stage names and the summed device
 * time, *steps the number of steps accumulated. */
int dvfe_profile(dvfe_tracker* t, int enable);
int dvfe_profile_read(dvfe_tracker* t, const char** names, double* total_ms, long* steps);

/* ---- the frame step ----------------------------------------------------------------- */

/* FeatureTracker::TrackImage(SemanticImage&) for all B streams (front_end/background_tracker.cpp:52-158).
 * left/right: HOST pointers (pinned or pageable) to stream 0's gray0/gray1 (CV_8UC1, `pitch` bytes per row);
 * stream s is at + s*stream_stride.  right may be NULL (mono frame).  time0[s] = SemanticImage::time0.
 * The call uploads the images, runs the whole step on the device and returns when the outputs are on
 * the host (read them with dvfe_get_features). */
int dvfe_track_image(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, size_t stream_stride, int pitch,
                     const double* time0);

/* Pipelined form of dvfe_track_image: uploads and enqueues the step and returns without waiting.  Up to two steps
 * may be in flight, so the host-to-device copy of frame k+1 overlaps the kernels of frame k (the call blocks only
 * while two earlier steps are still unfinished).  dvfe_wait() blocks until the OLDEST unfinished step is done and
 * makes its records the ones dvfe_get_features returns.  `left`/`right` must stay valid until that step is waited
 * for.  dvfe_track_image == dvfe_track_image_async + dvfe_wait. */
int dvfe_track_image_async(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, size_t stream_stride, int pitch,
                           const double* time0);
int dvfe_wait(dvfe_tracker* t);

/* Same step with the images already resident in device memory (no H2D inside). */
int dvfe_track_image_device(dvfe_tracker* t, const uint8_t* d_left, const uint8_t* d_right, size_t stream_stride,
                            int pitch, const double* time0);

/* Pipelined form of dvfe_track_image_device (pair with dvfe_wait): the D2H of step k and the host turn-around overlap
 * the kernels of step k+1.  The device images must stay unchanged until the step is waited for. */
int dvfe_track_image_device_async(dvfe_tracker* t, const uint8_t* d_left, const uint8_t* d_right, size_t stream_stride,
                                  int pitch, const double* time0);

/* Per-stream frame presence: one TrackImage step (enqueued, pair with dvfe_wait) in which every stream s gets exactly what a
 * single-stream tracker fed only that stream's frames would get.  stream_flags[s] (NULL = all 0):
 *   0                    the stream's frame as dvfe_track_image_async / dvfe_track_image_device_async (same graph, same launches
 *                        when every flag is 0)
 *   DVFE_FRAME_SKIP      no frame for this stream: FeatureTracker::TrackImage is not called.  Points, ids, next_id, track_cnt,
 *                        both velocity maps, prev_time and the previous-frame pyramid stay as they were; dvfe_get_features
 *                        returns 0 records; time0[s] is not read (NaN is fine)
 *   DVFE_FRAME_NO_RIGHT  left image only (TrackImage with an empty gray1, background_tracker.cpp:107): left points kept, no
 *                        cam-1 records, right_prev_* unchanged
 *   DVFE_FRAME_RESET     the stream starts over: before the frame it gets the state of a newly created tracker (n = 0,
 *                        next_id = 1, prev_time = 0) and the frame runs as a first frame; may be combined with NO_RIGHT
 * Unknown bits, SKIP|RESET and unknown `flags` bits return DVFE_ERR_INVALID and change nothing.  With right != NULL all B
 * slots of both images must be readable; the pixels of a skipped stream, and of a NO_RIGHT stream's right image, affect no
 * result.  right == NULL makes every stream mono.  flags: DVFE_STEP_DEVICE_INPUT = left / right are device pointers. */
#define DVFE_FRAME_SKIP 1u
#define DVFE_FRAME_NO_RIGHT 2u
#define DVFE_FRAME_RESET 4u
#define DVFE_STEP_DEVICE_INPUT 1u
int dvfe_track_image_ex(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, size_t stream_stride, int pitch,
                        const double* time0, const uint8_t* stream_flags, unsigned flags);

/* Backward-pass depth and forward-backward threshold of the LK at each of the reference's four call sites.  The
 * reference uses two pairs: the CPU FeatureTrackByLK (front_end/feature_utils.cpp:35-69: backward maxLevel 1, round
 * trip <= 0.5 px) and the cv::cuda call pattern of FeatureTrackByLKGpu (:83-163 with the objects created at
 * front_end/background_tracker.cpp:36-38: backward over all 3 levels, <= 1.0 px).  Defaults follow the reference:
 *   DVFE_LK_RAW_TEMPORAL, DVFE_LK_RAW_STEREO        TrackImage (:61-63, :117-118)                 CPU pair (1, 0.5)
 *   DVFE_LK_SEMANTIC_TEMPORAL                       TrackSemanticImage -> bg.TrackLeft (:783)      CPU pair (1, 0.5)
 *   DVFE_LK_SEMANTIC_STEREO                         TrackSemanticImage -> bg.TrackRightGPU (:801)  GPU pair (3, 1.0)
 * Both pairs are evaluated with this library's fixed-point LK arithmetic (cv::cuda's fp32 texture interpolation is not
 * reproduced).  dvfe_set_lk_mode_site sets one site; dvfe_set_lk_mode sets all four (e.g. (3, 1.0) for the
 * TrackImageNaive flow, front_end/background_tracker.cpp:400-516).  Applies to all later steps of the tracker. */
#define DVFE_LK_RAW_TEMPORAL 0
#define DVFE_LK_RAW_STEREO 1
#define DVFE_LK_SEMANTIC_TEMPORAL 2
#define DVFE_LK_SEMANTIC_STEREO 3
int dvfe_set_lk_mode(dvfe_tracker* t, int back_max_level, double fb_threshold);
int dvfe_set_lk_mode_site(dvfe_tracker* t, int site, int back_max_level, double fb_threshold);

/* Which detector InstFeat::DetectNewFeature (front_end/instance_feature.cpp:352-392) of the background uses in the semantic path:
 *   DVFE_DETECT_CPU   cv::goodFeaturesToTrack (use_gpu = false: TrackSemanticImage, front_end/background_tracker.cpp:789); default
 *   DVFE_DETECT_CUDA  DetectShiTomasiCornersGpu (use_gpu = true: TrackImageNaive, :445; front_end/feature_utils.cpp:339-348), i.e.
 *                     cv::cuda::GoodFeaturesToTrackDetector: the quality threshold is 0.01 x the maximum of the WHOLE response
 *                     map (cuda::minMax without the mask; the CPU detector takes the maximum over the unmasked pixels); candidates,
 *                     ordering and the distance grid are the same.  Evaluated with this library's CPU-parity response arithmetic
 *                     (cv::cuda's fp32 box sums are not reproduced; its candidate buffer of max(1000, 5 % of the pixels) entries
 *                     is not modelled either).
 * TrackImageNaive = dvfe_set_lk_mode_site(t, DVFE_LK_SEMANTIC_TEMPORAL and _STEREO, 3, 1.0) + dvfe_set_detect_mode(t,
 * DVFE_DETECT_CUDA) + dvfe_track_semantic_image; the host wrappers (include/dvfe/feature_tracker.hpp, dynamic_vins_b200/tracker.py)
 * put the caller's modes back before the next call of another entry point. */
#define DVFE_DETECT_CPU 0
#define DVFE_DETECT_CUDA 1
int dvfe_set_detect_mode(dvfe_tracker* t, int mode);

/* FeatureTracker::TrackSemanticImage(SemanticImage&) (front_end/background_tracker.cpp:757-837).
 * inv_merge_mask: HOST, same layout as left (0 = object, 255 = background), may be NULL when no stream has
 * instances; exist_inst[s] = SemanticImage::exist_inst. */
int dvfe_track_semantic_image(dvfe_tracker* t, const uint8_t* left, const uint8_t* right,
                              const uint8_t* inv_merge_mask, size_t stream_stride, int pitch,
                              const int* exist_inst, const double* time0);

/* Per-stream frame presence for TrackSemanticImage (and TrackImageNaive, see dvfe_set_detect_mode): one step, enqueued (pair with
 * dvfe_wait), in which every stream s gets exactly what a single-stream tracker fed only that stream's frames would get.
 * stream_flags[s] as for dvfe_track_image_ex (NULL or all 0: the step dvfe_track_semantic_image enqueues, same graph, same
 * launches); a skipped stream's exist_inst[s], mask and time0[s] are not read.  DVFE_FRAME_RESET also starts the stream's
 * instance manager over (as dvfe_track_dynamic_ex2).  A following dvfe_insts_track / dvfe_insts_track_batch of the same frame
 * obeys the flags: a skipped stream must have 0 boxes and is left untouched, a DVFE_FRAME_NO_RIGHT stream's instances run mono.
 * flags: DVFE_DYN_DEVICE_INPUT (left / right / mask are device pointers) only.  Invalid stream flags and unknown `flags` bits
 * return DVFE_ERR_INVALID and change nothing.  dvfe_track_semantic_image == wait for all steps + this with NULL flags + wait. */
int dvfe_track_semantic_ex(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, const uint8_t* inv_merge_mask,
                           size_t stream_stride, int pitch, const int* exist_inst, const double* time0,
                           const uint8_t* stream_flags, unsigned flags);

/* InstsFeatManager::InstsTrack(SemanticImage) preceded by the caller's per-frame instance reset and
 * AddViodeInstances (system/main.cpp:198-210, front_end/dynamic_tracker.cpp:348-493,585-605), for ONE stream.
 * Uses the gray0/gray1 uploaded by the last dvfe_track_semantic_image call of that stream. */
int dvfe_insts_track(dvfe_tracker* t, int stream, const dvfe_inst_in* insts, int n_insts, double time0);

/* The same for ALL streams of the tracker in one set of launches: `insts` holds the boxes stream by stream
 * (n_insts[0] boxes of stream 0, then n_insts[1] of stream 1, ...), time0[s] per stream. */
int dvfe_insts_track_batch(dvfe_tracker* t, const dvfe_inst_in* insts, const int* n_insts, const double* time0);

/* One frame of dynamic mode for all streams, enqueued (pair with dvfe_wait): TrackSemanticImage + the caller's per-frame
 * instance reset + AddViodeInstances + InstsTrack (system/main.cpp:193-254).  dvfe_track_dynamic_async is the flags = 0 form.
 *   DVFE_DYN_DEVICE_INPUT  left / right / mask are DEVICE pointers (frames decoded or rendered on the GPU): nothing is uploaded
 *   DVFE_DYN_LABELS        SemanticImage::SetMaskAndRoi on the device (basic/semantic_image.cpp:20-63): `mask` is ONE label image
 *                          per stream (u8, layout of `left` at 1 byte/px) in which bit b of a pixel says that the pixel belongs
 *                          to the instance whose box carries label_bit == b (up to 8 instances per frame, overlaps allowed).
 *                          inv_merge_mask (no bit set -> 255) and every box's ROI mask full_mask(rect) are derived on the device;
 *                          the per-box host masks and the inv_merge_mask upload disappear. */
#define DVFE_DYN_DEVICE_INPUT 1u
#define DVFE_DYN_LABELS 2u
int dvfe_track_dynamic_ex(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, const uint8_t* mask, size_t stream_stride,
                          int pitch, const int* exist_inst, const dvfe_inst_in* boxes, const int* n_boxes, const double* time0,
                          unsigned flags);

/* dvfe_track_dynamic_ex with per-stream frame presence (dvfe_track_dynamic_ex and dvfe_track_dynamic_async are this with
 * stream_flags = NULL).  stream_flags[s] (NULL or all 0: the plain step, same graph, same launches):
 *   DVFE_FRAME_SKIP      neither TrackSemanticImage nor InstsTrack is called for the stream: the background as for
 *                        dvfe_track_image_ex; no per-frame instance reset, no lost_num change, no ManageInstances, last_time and the
 *                        ROI buffers kept; dvfe_get_features and dvfe_insts_output return 0 records, dvfe_insts_table is unchanged.
 *                        n_boxes[s] must be 0; the stream's pixels, mask / label image, exist_inst[s] and time0[s] are not read
 *   DVFE_FRAME_NO_RIGHT  a mono frame for the stream: no cam-1 records for the background or the instances, no TrackRightByPad,
 *                        the right velocity maps kept
 *   DVFE_FRAME_RESET     a newly created FeatureTracker and InstsFeatManager for the stream (no points, next_id = 1 before the
 *                        background detection, prev_time = 0; no instances, every slot free, last_time = 0); boxes allowed (they are
 *                        the new manager's first frame); may be combined with NO_RIGHT
 * Unknown bits, SKIP|RESET and boxes for a skipped stream return DVFE_ERR_INVALID and change nothing. */
int dvfe_track_dynamic_ex2(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, const uint8_t* mask, size_t stream_stride,
                           int pitch, const int* exist_inst, const dvfe_inst_in* boxes, const int* n_boxes, const double* time0,
                           const uint8_t* stream_flags, unsigned flags);

/* FeatureBackground of stream s of the last step: n_out records, sorted by (id, cam). */
int dvfe_get_features(dvfe_tracker* t, int stream, dvfe_obs* out, int cap, int* n_out);
/* InstsFeatManager::Output() (front_end/dynamic_tracker.cpp:521-577), sorted by (inst_id, id). */
int dvfe_insts_output(dvfe_tracker* t, int stream, dvfe_inst_obs* out, int cap, int* n_out);

/* The instance table after the last InstsTrack of a stream: InstsFeatManager::instances (front_end/dynamic_tracker.h:83)
 * with the fields the caller's per-frame code reads (system/main.cpp:198-242: is_curr_visible, box2d) and the bookkeeping
 * ManageInstances keeps (lost_num, front_end/dynamic_tracker.cpp:499-514).  Rows in ascending track id. */
typedef struct dvfe_inst_info {
    uint32_t track_id;
    int32_t lost_num;
    int32_t is_curr_visible;
    int32_t has_box;            /* box2d != nullptr */
    int32_t x, y, w, h;         /* box2d->rect of the last frame the instance was seen in */
} dvfe_inst_info;
int dvfe_insts_table(dvfe_tracker* t, int stream, dvfe_inst_info* out, int cap, int* n_out);

/* ---- tracker state (InstFeat bg members, front_end/instance_feature.h:103-137) --------------- */
typedef struct dvfe_state {
    int n;                      /* bg.ids.size() */
    uint32_t next_id;           /* InstFeat::global_id_count */
    double prev_time;
    uint32_t* ids;              /* [cap] bg.ids */
    int32_t* track_cnt;         /* [cap] bg.track_cnt */
    float* last_points;         /* [cap*2] bg.last_points (= curr_points of the last frame) */
    float* prev_un;             /* [cap*2] bg.prev_id_pts values, in ids order */
    float* right_prev_un;       /* [cap*2] bg.right_prev_id_pts values (valid where right_prev_valid) */
    uint8_t* right_prev_valid;  /* [cap] */
} dvfe_state;
/* dvfe_get_state / dvfe_set_state cover the background point arrays of one stream (what the teacher-forced parity tests
 * exchange with the oracle), NOT the previous-frame pyramid nor the instance table / ROI buffers: set_state is valid on a tracker
 * that has already processed the previous frame (its pyramid is the LK template image of the next step); on a fresh tracker
 * (no frame yet) the next step has no previous image and treats the restored points as the first frame's.  set_state
 * invalidates the LK template caches and the captured step graphs. */
int dvfe_get_state(dvfe_tracker* t, int stream, dvfe_state* st, int cap);
int dvfe_set_state(dvfe_tracker* t, int stream, const dvfe_state* st);

/* ---- seam-level operators (unit parity; each replaces one OpenCV/camodocal call of the path) ---- */

/* cv::buildOpticalFlowPyramid(img, pyr, Size(21,21), max_level) as used inside calcOpticalFlowPyrLK.
 * Writes level l (l = 0..*n_levels-1) unpadded into out_levels[l] (size ((w+1)/2.., (h+1)/2..)). */
int dvfe_op_build_pyramid(const uint8_t* img, int w, int h, int pitch, int max_level, uint8_t* const* out_levels,
                          int* level_w, int* level_h, int* n_levels);
/* One level of the same pyramid WITH its border, as cv::buildOpticalFlowPyramid(img, pyr, winSize, maxLevel, false,
 * BORDER_REFLECT_101) stores it: out = dense (w_l + 2 border) x (h_l + 2 border) bytes, border <= 21 (= winSize).  The LK
 * kernels read this border; levels >= 1 write it from the down-sampling kernel itself. */
int dvfe_op_build_pyramid_bordered(const uint8_t* img, int w, int h, int pitch, int max_level, int level, int border,
                                   uint8_t* out);

/* FeatureTrackByLK(img1,img2,pts1,pts2,flow_back) (front_end/feature_utils.cpp:35-69):
 * forward LK (max_level) + backward LK (max level 1, initial flow) + 0.5 px check + InBorder.
 * mask (nullable, same size as the images): status also cleared where mask[cvRound(pt2)] == 0
 * (InstFeat::TrackLeft, front_end/instance_feature.cpp:166-171).  pts are (x,y) float pairs.
 * rev_out (nullable): backward-tracked points. */
int dvfe_op_lk(const uint8_t* img1, const uint8_t* img2, int w, int h, int pitch, const float* pts1, int n,
               int flow_back, int max_level, const uint8_t* mask, int mask_pitch, float* pts2_out,
               uint8_t* status_out, float* rev_out);

/* cv::cornerMinEigenVal(img, eig, 3, 3) — the response map of goodFeaturesToTrack. */
int dvfe_op_min_eigen_val(const uint8_t* img, int w, int h, int pitch, float* eig_out);

/* cv::goodFeaturesToTrack(img, corners, max_corners, quality, min_dist, mask)
 * (front_end/background_tracker.cpp:85, front_end/instance_feature.cpp:381, front_end/dynamic_tracker.cpp:435).
 * eig (nullable): use this response map instead of computing it (NMS parity "given equal response maps"). */
int dvfe_op_good_features(const uint8_t* img, int w, int h, int pitch, const float* eig, const uint8_t* mask,
                          int mask_pitch, int max_corners, double quality, double min_dist, float* corners_out,
                          int* n_out, int* n_candidates_out);

/* for each pt: cv::circle(mask, pt, radius, 0, -1) (front_end/background_tracker.cpp:79-80). In place. */
/* The same with the cv::cuda detector's threshold (DVFE_DETECT_CUDA above): DetectShiTomasiCornersGpu, front_end/feature_utils.cpp:339-348. */
int dvfe_op_good_features_cuda(const uint8_t* img, int w, int h, int pitch, const float* eig, const uint8_t* mask,
                               int mask_pitch, int max_corners, double quality, double min_dist, float* corners_out,
                               int* n_out, int* n_candidates_out);
int dvfe_op_disc_mask(uint8_t* mask, int w, int h, int pitch, const float* pts, int n, int radius);

/* ErodeMask(in,out,k): cv::erode with a k x k MORPH_RECT element (front_end/feature_utils.h:142-146). */
int dvfe_op_erode_rect(const uint8_t* src, int w, int h, int pitch, int k, uint8_t* dst);

/* InstFeat::UndistortedPts / UndistortedPointsWithAddOffset: PinholeCamera::liftProjective then (x/z, y/z)
 * narrowed to float (front_end/instance_feature.cpp:94-103,123-133). */
int dvfe_op_lift_projective(const dvfe_camera* cam, const float* pts, int n, float off_x, float off_y, float* out);

/* ---- upstream frame preparation (SURVEY.md §8f N1) ----------------------------------------------------- */

/* SemanticImage::SetGrayImage: cv::cvtColor(color, gray, CV_BGR2GRAY) (basic/semantic_image.cpp:69-73).
 * bgr: h rows of 3*w bytes (pitch bytes per row) -> gray_out: dense w x h. */
int dvfe_op_bgr_to_gray(const uint8_t* bgr, int w, int h, int pitch, uint8_t* gray_out);

/* SemanticImage::SetMaskAndRoi / SetBackgroundMask (basic/semantic_image.cpp:20-63,103-117): masks = n dense w x h
 * instance masks (non-zero = object) -> merge_mask (255 = object) and inv_merge_mask (bitwise_not). */
int dvfe_op_merge_masks(const uint8_t* masks, int n_masks, int w, int h, uint8_t* merge_out, uint8_t* inv_out);

/* FeatureTrack() static-instance punch-out (system/main.cpp:219-242): merge_mask = 0 (and inv_merge_mask = 255) wherever the
 * ROI mask (roi_h x roi_w at rect.tl() = (x, y)) of a static instance is set.  Both full masks are dense w x h, in place. */
int dvfe_op_punch_out(uint8_t* merge_mask, uint8_t* inv_merge_mask, int w, int h, const uint8_t* roi_mask, int roi_pitch,
                      int x, int y, int roi_w, int roi_h);

/* ImageProcessor::Run undistortion (image_process/image_process.cpp:109-122): cv::remap(src, dst, map1, map2, INTER_LINEAR)
 * with the fixed-point maps of cv::initUndistortRectifyMap(..., CV_16SC2, map1, map2) (utils/camera_model.cpp:483-497):
 * map1 = w*h (x, y) int16 pairs, map2 = w*h uint16 table indices; BORDER_CONSTANT 0; dst has the size of src.
 * channels 1 | 3.  to_gray != 0 with 3 channels additionally applies cvtColor(BGR2GRAY) (dst = dense w x h);
 * otherwise dst = dense w x h x channels.  map1 == map2 == NULL: identity (only the gray conversion runs). */
int dvfe_op_remap(const uint8_t* src, int w, int h, int channels, int pitch, const int16_t* map1, const uint16_t* map2,
                  int to_gray, uint8_t* dst);

/* One frame of dynamic mode for ALL streams, pipelined (the asynchronous form of FeatureTrack()'s dynamic branch,
 * system/main.cpp:247-254: TrackSemanticImage + InstsTrack of the same frame): both are enqueued behind the previous
 * step (two steps in flight; the uploads of frame k+1 overlap the kernels of frame k) and the call returns.
 * dvfe_wait() completes the oldest step; dvfe_get_features / dvfe_insts_output then return ITS results.
 * Arguments as dvfe_track_semantic_image + dvfe_insts_track_batch; the images, masks and ROI masks must stay valid until
 * the matching dvfe_wait() (ROI masks are copied to a staging buffer during the call when they fit it). */
int dvfe_track_dynamic_async(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, const uint8_t* inv_merge_mask,
                             size_t stream_stride, int pitch, const int* exist_inst, const dvfe_inst_in* boxes,
                             const int* n_boxes, const double* time0);

/* ---- frame ingest inside the tracker (SURVEY.md §8f N1 + N2) ---------------------------------------------
 * dvfe_set_input: the images handed to dvfe_track_image[_async|_device*] / dvfe_track_semantic_image are `channels`
 * interleaved bytes per pixel: 1 = gray (default), 3 = BGR as in SemanticImage::color0/color1; pitch >= channels * width.
 * dvfe_set_undistort_maps: cfg::is_undistort_input — every image of camera `cam` (0 left, 1 right) is first remapped
 * through (map1, map2) as cv::remap does (see dvfe_op_remap); the maps are copied to the device and shared by all
 * streams; (NULL, NULL) clears them.  Both run on the device, fused into one pass that writes pyramid level 0:
 * gray0 = cvtColor(remap(color0)) is never materialised on the host.  The region mask of
 * dvfe_track_semantic_image is NOT remapped (the caller passes SetBackgroundMask's result, basic/semantic_image.cpp:103-117)
 * and stays one byte per pixel: with a 3-channel input its row pitch is pitch / 3 and its stream stride stream_stride / 3. */
int dvfe_set_input(dvfe_tracker* t, int channels);
int dvfe_set_undistort_maps(dvfe_tracker* t, int cam, const int16_t* map1, const uint16_t* map2);

/* ---- epipolar outlier rejection and extra points (SURVEY.md §8f N4) --------------------------------------
 * InstsFeatManager::RejectWithF (front_end/dynamic_tracker.cpp:831-849; FeatureTracker::RejectWithF,
 * front_end/background_tracker.cpp:520-550, is the same call): cur_pts / prev_pts are n distorted pixel positions (x, y);
 * both are lifted with `cam` (PinholeCamera::liftProjective), re-projected with kFocalLength = 460 about (col/2, row/2),
 * narrowed to float and given to cv::findFundamentalMat(cur, prev, FM_RANSAC, f_threshold, 0.99, status).
 * status[n] receives the inlier bytes; *n_status = n, or 0 when n < 7 (OpenCV then leaves `status` empty).  The sample order
 * is that of cv::RNG(-1), the 7-point models are solved in fp64; see dynamic_vins_b200/csrc/geometry.cu for what is and is not
 * reproducible about OpenCV's null-space basis (ties between roots of one sample, LMedS with 8 <= n <= 13). */
int dvfe_op_reject_with_f(const dvfe_camera* cam, const float* cur_pts, const float* prev_pts, int n, int col, int row,
                          double f_threshold, uint8_t* status, int* n_status);

/* InstFeat::DetectExtraPoints (front_end/instance_feature.cpp:413-461): samples the ROI mask (rows x cols, box2d->rect.tl() =
 * (box_x, box_y)) on the reference's grid (step = max(sqrt(0.8*rows*cols/1000), 2)), reads the CV_32F disparity map at the
 * full-image position and emits (x, y, depth) = ((c-cx)*depth/fx, (r-cy)*depth/fy, fx*baseline/disparity) for samples with
 * mask != 0, disparity > 0 and not NaN, 0.1 < depth <= 100 (float arithmetic, CameraInfo's float intrinsics), in row-major sample
 * order.  out = 3 doubles per point (extra_points3d is a vector<Vec3d>), cap points; *n_out = the count (DVFE_ERR_CAPACITY if
 * it exceeds cap). */
int dvfe_op_detect_extra_points(const uint8_t* roi_mask, int rows, int cols, int mask_pitch, const float* disp, int disp_w,
                                int disp_h, int disp_pitch, int box_x, int box_y, float fx, float fy, float cx, float cy,
                                float baseline, double* out, int cap, int* n_out);

#ifdef __cplusplus
}
#endif
#endif /* DVFE_H_ */
