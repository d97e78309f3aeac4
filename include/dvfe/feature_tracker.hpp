// C++ host mirror of the reference's front-end classes over the C ABI (include/dvfe.h).
//
// Same class names, member names, argument meaning and error behaviour as
//   dynamic_vins::FeatureTracker    dynamic_vins/src/front_end/background_tracker.h:40-89
//   dynamic_vins::InstsFeatManager  dynamic_vins/src/front_end/dynamic_tracker.h:40-100
//   SemanticImage / Box2D / InstRoi / FeatureBackground / FeatureInstance / FeaturePoint
//                                   basic/semantic_image.h:29-66, basic/box2d.h:24-56, basic/frontend_feature.h:34-73,
//                                   basic/point_feature.h:22-100
// with the OpenCV / Eigen types replaced by plain views so that the header has no dependency:
//   cv::Mat (CV_8UC1 / CV_32FC1)           -> GrayImage / FloatImage {data, rows, cols, step}   (views, no ownership)
//   cv::Rect2f, cv::Point2f, cv::Scalar    -> Rect2f, Point2f, Scalar
//   Eigen::Matrix<double,7,1> (Vec7d)      -> std::array<double,7>   (layout compatible: 7 contiguous doubles)
//   Eigen::Vector3d / Vector2d             -> std::array<double,3> / <double,2>
// Call sequence of one frame, as FeatureTrack() drives it (system/main.cpp:178-330):
//   raw mode      frame.features = feature_tracker->TrackImage(*img);
//   dynamic mode  for (auto& [id, inst] : insts_tracker->instances) { inst.is_curr_visible = false; inst.box2d.reset(); }
//                 insts_tracker->AddViodeInstances(*img);
//                 frame.features  = feature_tracker->TrackSemanticImage(*img);     // the reference runs these two on two
//                 insts_tracker->InstsTrack(*img);                                 // threads racing for the id counter;
//                 frame.instances = insts_tracker->Output();                       // here: background first (DESIGN.md Q5)
// The reference throws std::runtime_error for a bad settings path or empty input; so does this mirror (the C ABI underneath
// returns codes).  Header only; link with -ldvfe.
#pragma once
#include <array>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../dvfe.h"
#include "reject_with_f.h"

namespace dynamic_vins {

using Vec7d = std::array<double, 7>;
using Vec3d = std::array<double, 3>;
using Vec2d = std::array<double, 2>;

struct GrayImage {                       // a CV_8UC1 (or, for BGR input, CV_8UC3) cv::Mat header
    const uint8_t* data = nullptr;
    int rows = 0, cols = 0, step = 0;
    bool empty() const { return data == nullptr || rows == 0 || cols == 0; }
};
struct FloatImage {                      // a CV_32FC1 cv::Mat header (SemanticImage::disp)
    const float* data = nullptr;
    int rows = 0, cols = 0, step = 0;    // step in bytes
    bool empty() const { return data == nullptr || rows == 0 || cols == 0; }
};
struct Point2f { float x = 0, y = 0; };
struct Rect2f {                          // cv::Rect2f
    float x = 0, y = 0, width = 0, height = 0;
    Point2f tl() const { return {x, y}; }
    Point2f br() const { return {x + width, y + height}; }
};
using Scalar = std::array<double, 4>;    // cv::Scalar

struct InstRoi {                         // basic/box2d.h:24-36 (the host-side members)
    using Ptr = std::shared_ptr<InstRoi>;
    GrayImage mask_cv;                   // rect-sized, 255 = object
    GrayImage roi_gray;                  // rect-sized crop of gray0 (the library crops it on the device; kept for shape parity)
};

struct Box2D {                           // basic/box2d.h:39-56
    using Ptr = std::shared_ptr<Box2D>;
    std::string class_name;
    int class_id = 0, id = 0, track_id = 0;
    Point2f min_pt, max_pt;
    Rect2f rect;
    float score = 0.f;
    InstRoi::Ptr roi;
    Point2f center_pt() const { return {(min_pt.x + max_pt.x) / 2.f, (min_pt.y + max_pt.y) / 2.f}; }
};

struct SemanticImage {                   // basic/semantic_image.h:29-66 (the members the front-end reads)
    GrayImage color0, color1;            // only their size is read by the reference's front-end
    GrayImage gray0, gray1;
    double time0 = 0.0, time1 = 0.0;
    unsigned int seq = 0;
    GrayImage merge_mask;                // 255 = object
    GrayImage inv_merge_mask;            // 0 = object, 255 = background
    FloatImage disp;                     // optional disparity map (Output() reads it, reference quirk Q8)
    bool exist_inst = false;
    std::vector<Box2D::Ptr> boxes2d;
};

struct FeatureBackground {               // basic/frontend_feature.h:34-47
    std::map<unsigned int, std::vector<std::pair<int, Vec7d>>> points;
};

struct FeaturePoint {                    // basic/point_feature.h:22-100
    using Ptr = std::shared_ptr<FeaturePoint>;
    Vec3d point{0, 0, 0}, point_right{0, 0, 0};
    bool is_stereo = false, is_extra = false;
    int frame = 0;
    Vec2d vel{0, 0}, vel_right{0, 0};
    double td = 0;
    float disp = 0.f;
};

struct FeatureInstance {                 // basic/frontend_feature.h:49-58
    std::map<unsigned int, FeaturePoint::Ptr> features;
    Scalar color{0, 0, 0, 0};
    Box2D::Ptr box2d;
    std::shared_ptr<void> box3d;         // 3-D detection boxes are outside this path: always null
    std::vector<Vec3d> points;           // extra (PCL) points are outside this path: always empty
};

struct FrontendFeature {                 // basic/frontend_feature.h:64-73: what the front-end hands to the estimator
    FeatureBackground features;
    double time = 0.0;
    unsigned int seq_id = 0;
    std::map<unsigned int, FeatureInstance> instances;
};

// One detected / tracked object as InstsFeatManager keeps it (front_end/instance_feature.h:103-137: the members the
// caller's per-frame code touches).  Points, velocities and ROI images live on the device.
struct InstFeat {
    unsigned int id = 0;
    Scalar color{0, 0, 0, 0};
    int lost_num = 0;
    bool is_curr_visible = false;
    Box2D::Ptr box2d;
    std::shared_ptr<void> box3d;
    InstRoi::Ptr roi = std::make_shared<InstRoi>();
};

struct InstEstimatedInfo {               // basic/inst_estimated_info.h (the flag the caller's punch-out reads)
    bool is_init = false, is_static = false;
    double time = 0.0;
};

class InstsFeatManager;

class FeatureTracker {
public:
    using Ptr = std::unique_ptr<FeatureTracker>;
    // FeatureTracker(const string& config_path): fe_para::SetParameters + the camera yaml files.  max_instances > 0 also
    // allocates the per-instance state an InstsFeatManager attached to this tracker needs (slam_type "dynamic" does so too).
    explicit FeatureTracker(const std::string& config_path, int device = 0, int max_instances = -1) : config_path_(config_path) {
        if (dvfe_config_from_yaml(config_path.c_str(), &cfg_) != DVFE_OK) throw std::runtime_error(dvfe_last_error(nullptr));
        cfg_.device = device;
        if (max_instances >= 0) cfg_.max_instances = max_instances;
        if (dvfe_create(&cfg_, &h_) != DVFE_OK) throw std::runtime_error(dvfe_last_error(nullptr));
        current() = this;
    }
    explicit FeatureTracker(const dvfe_config& cfg) : cfg_(cfg) {
        if (dvfe_create(&cfg_, &h_) != DVFE_OK) throw std::runtime_error(dvfe_last_error(nullptr));
        current() = this;
    }
    ~FeatureTracker() {
        if (current() == this) current() = nullptr;
        dvfe_destroy(h_);
    }
    FeatureTracker(const FeatureTracker&) = delete;
    FeatureTracker& operator=(const FeatureTracker&) = delete;

    // front_end/background_tracker.cpp:52-158
    FeatureBackground TrackImage(SemanticImage& img) {
        check_input(img);
        leave_naive();
        cur_img = img;
        const bool right = cfg_.stereo && !img.gray1.empty();
        if (dvfe_track_image(h_, img.gray0.data, right ? img.gray1.data : nullptr, (size_t)img.gray0.step * img.gray0.rows,
                             img.gray0.step, &img.time0) != DVFE_OK)
            throw std::runtime_error(dvfe_last_error(h_));
        prev_img = cur_img;
        return SetOutputFeats();
    }
    // front_end/background_tracker.cpp:757-837
    FeatureBackground TrackSemanticImage(SemanticImage& img) {
        leave_naive();
        return semantic(img);
    }
    // FeatureTracker::TrackImageNaive (:400-516): the cv::cuda flow — ErodeMaskGpu, TrackLeftGPU, DetectNewFeature(use_gpu),
    // TrackRightGPU — i.e. the cv::cuda call pattern (3, 1.0) at both semantic LK sites and the cv::cuda detector's threshold rule,
    // evaluated with this library's CPU-parity arithmetic; the dynamic regions are removed through inv_merge_mask like
    // TrackSemanticImage does.  These modes hold for the naive calls only: the next TrackImage / TrackSemanticImage runs with the
    // modes set through SetLkMode / SetDetectMode (the library's defaults unless changed).
    FeatureBackground TrackImageNaive(SemanticImage& img) {
        if (!naive_mode_) {
            set_lk_site(DVFE_LK_SEMANTIC_TEMPORAL, 3, 1.0);
            set_lk_site(DVFE_LK_SEMANTIC_STEREO, 3, 1.0);
            if (dvfe_set_detect_mode(h_, DVFE_DETECT_CUDA) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
            naive_mode_ = true;
        }
        return semantic(img);
    }
    // dvfe_set_lk_mode_site / dvfe_set_detect_mode for the TrackImage and TrackSemanticImage calls of this tracker (site -1: all four)
    void SetLkMode(int back_max_level, double fb_threshold, int site = -1) {
        leave_naive();
        if (dvfe_set_lk_mode_site(h_, site, back_max_level, fb_threshold) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
        for (int i = 0; i < 4; i++)
            if (site < 0 || site == i) lk_[i] = {back_max_level, fb_threshold};
    }
    void SetDetectMode(bool cuda_semantics) {
        leave_naive();
        if (dvfe_set_detect_mode(h_, cuda_semantics ? DVFE_DETECT_CUDA : DVFE_DETECT_CPU) != DVFE_OK)
            throw std::runtime_error(dvfe_last_error(h_));
        detect_cuda_ = cuda_semantics;
    }
    // FeatureTracker::RejectWithF inside every background step (dvfe_set_reject_with_f): f_threshold = fe_para::F_threshold
    // (dvfe_f_threshold_from_yaml), 0 = off.  The constructor leaves it off, as the reference's TrackImage never calls it.
    void SetRejectWithF(double f_threshold) {
        if (dvfe_set_reject_with_f(h_, f_threshold) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
    }
    // visualisation (DrawTrack) is outside the path: the image stays empty, the accessor exists for source compatibility
    GrayImage& img_track() { return img_vis_; }

    // ImageProcessor::Run moved onto the device (image_process/image_process.cpp:105-126): with SetColorInput(true) the
    // gray0/gray1 views of SemanticImage carry color0/color1 (BGR, step >= 3 * cols; inv_merge_mask stays 1 byte/px
    // with step = color step / 3); SetUndistortMaps hands over cam_s.left/right_undist_map1/2 (CV_16SC2 + CV_16UC1,
    // utils/camera_model.cpp:483-497) and every image of that camera is remapped before the gray conversion.
    void SetColorInput(bool bgr) {
        if (dvfe_set_input(h_, bgr ? 3 : 1) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
        channels_ = bgr ? 3 : 1;
    }
    void SetUndistortMaps(int cam, const int16_t* map1, const uint16_t* map2) {
        if (dvfe_set_undistort_maps(h_, cam, map1, map2) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
    }
    dvfe_tracker* handle() { return h_; }
    const dvfe_config& config() const { return cfg_; }
    const std::string& config_path() const { return config_path_; }

    SemanticImage prev_img, cur_img;     // background_tracker.h:49 (views of the caller's buffers)

    // The reference shares one process-global feature-id counter (InstFeat::global_id_count) between its FeatureTracker
    // and its InstsFeatManager; here both live in one dvfe_tracker, which InstsFeatManager(config_path) finds here.
    static FeatureTracker*& current() { static FeatureTracker* cur = nullptr; return cur; }

private:
    // front_end/background_tracker.cpp:757-837 with the modes in force
    FeatureBackground semantic(SemanticImage& img) {
        check_input(img);
        cur_img = img;
        const bool right = cfg_.stereo && !img.gray1.empty();
        const int exist = img.exist_inst ? 1 : 0;
        if (img.exist_inst && (img.inv_merge_mask.empty() || img.inv_merge_mask.step != img.gray0.step / channels_))
            throw std::runtime_error("TrackSemanticImage: inv_merge_mask must have the layout of gray0");
        if (dvfe_track_semantic_image(h_, img.gray0.data, right ? img.gray1.data : nullptr,
                                      img.exist_inst ? img.inv_merge_mask.data : nullptr,
                                      (size_t)img.gray0.step * img.gray0.rows, img.gray0.step, &exist,
                                      &img.time0) != DVFE_OK)
            throw std::runtime_error(dvfe_last_error(h_));
        prev_img = cur_img;
        return SetOutputFeats();
    }
    void set_lk_site(int site, int back_max_level, double fb_threshold) {
        if (dvfe_set_lk_mode_site(h_, site, back_max_level, fb_threshold) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
    }
    // the caller's modes again at the two sites and the detector a naive call switched
    void leave_naive() {
        if (!naive_mode_) return;
        for (int site : {DVFE_LK_SEMANTIC_TEMPORAL, DVFE_LK_SEMANTIC_STEREO}) set_lk_site(site, lk_[site].first, lk_[site].second);
        if (dvfe_set_detect_mode(h_, detect_cuda_ ? DVFE_DETECT_CUDA : DVFE_DETECT_CPU) != DVFE_OK)
            throw std::runtime_error(dvfe_last_error(h_));
        naive_mode_ = false;
    }
    void check_input(const SemanticImage& img) const {
        if (img.gray0.empty() || img.gray0.cols != cfg_.width || img.gray0.rows != cfg_.height)
            throw std::runtime_error("FeatureTracker: gray0 is empty or does not match image_width/image_height");
    }
    // front_end/background_tracker.cpp:340-392
    FeatureBackground SetOutputFeats() {
        std::vector<dvfe_obs> rec(2 * (size_t)cfg_.max_cnt);
        int n = 0;
        if (dvfe_get_features(h_, 0, rec.data(), (int)rec.size(), &n) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
        FeatureBackground fm;
        for (int i = 0; i < n; i++) {
            Vec7d v;
            for (int k = 0; k < 7; k++) v[k] = rec[i].v[k];
            fm.points[rec[i].id].emplace_back(rec[i].cam, v);
        }
        return fm;
    }
    dvfe_config cfg_{};
    dvfe_tracker* h_ = nullptr;
    std::string config_path_;
    int channels_ = 1;
    bool naive_mode_ = false;                                            // the naive call pattern is switched on
    std::pair<int, double> lk_[4] = {{1, 0.5}, {1, 0.5}, {1, 0.5}, {3, 1.0}};    // SetLkMode per site (include/dvfe.h defaults)
    bool detect_cuda_ = false;                                           // SetDetectMode
    GrayImage img_vis_;
};

class InstsFeatManager {
public:
    using Ptr = std::shared_ptr<InstsFeatManager>;
    // front_end/dynamic_tracker.cpp:33-38.  The manager works on the device state of the process's FeatureTracker (created
    // before it from the same config, as in system/main.cpp:344-347).
    explicit InstsFeatManager(const std::string& config_path) : t_(*require_tracker(config_path)) {}
    explicit InstsFeatManager(FeatureTracker& tracker) : t_(tracker) {}

    // front_end/dynamic_tracker.cpp:585-605: the frame's detections arrive with track ids; visible instances take the box.
    void AddViodeInstances(SemanticImage& img) {
        for (auto& det_box : img.boxes2d) {
            const unsigned key = (unsigned)det_box->track_id;
            if (instances.count(key) == 0) { InstFeat f; f.id = key; instances.insert({key, f}); }
            InstFeat& inst = instances[key];
            inst.box2d = det_box;
            if (det_box->roi) { inst.roi->mask_cv = det_box->roi->mask_cv; inst.roi->roi_gray = det_box->roi->roi_gray; }
            inst.is_curr_visible = true;
        }
    }

    // front_end/dynamic_tracker.cpp:348-493 for the instances the caller marked visible (system/main.cpp:198-210).
    // Call after FeatureTracker::TrackSemanticImage of the same frame.
    void InstsTrack(SemanticImage img) {
        std::vector<dvfe_inst_in> in;
        for (auto& kv : sorted_instances()) {
            const InstFeat& inst = *kv.second;
            if (!inst.is_curr_visible || !inst.box2d) continue;
            const Box2D& b = *inst.box2d;
            dvfe_inst_in d{};
            d.track_id = kv.first;
            d.x = (int)b.rect.x; d.y = (int)b.rect.y; d.w = (int)b.rect.width; d.h = (int)b.rect.height;
            d.mask = inst.roi->mask_cv.data; d.mask_pitch = inst.roi->mask_cv.step;
            d.disp = img.disp.empty() ? nullptr : img.disp.data; d.disp_pitch = img.disp.step;
            in.push_back(d);
        }
        if (dvfe_insts_track(t_.handle(), 0, in.empty() ? nullptr : in.data(), (int)in.size(), img.time0) != DVFE_OK)
            throw std::runtime_error(dvfe_last_error(t_.handle()));
        sync_table();
        prev_img_ = img;
    }

    // front_end/dynamic_tracker.cpp:521-577
    std::map<unsigned int, FeatureInstance> Output() {
        const dvfe_config& c = t_.config();
        std::vector<dvfe_inst_obs> rec((size_t)(c.max_instances > 0 ? c.max_instances : 1) * (size_t)(c.max_dynamic_cnt > 0 ? c.max_dynamic_cnt : 1));
        int n = 0;
        if (dvfe_insts_output(t_.handle(), 0, rec.data(), (int)rec.size(), &n) != DVFE_OK)
            throw std::runtime_error(dvfe_last_error(t_.handle()));
        std::map<unsigned int, FeatureInstance> out;
        for (int i = 0; i < n; i++) {
            FeaturePoint::Ptr f = std::make_shared<FeaturePoint>();
            for (int k = 0; k < 3; k++) { f->point[k] = rec[i].point[k]; f->point_right[k] = rec[i].point_right[k]; }
            for (int k = 0; k < 2; k++) { f->vel[k] = rec[i].vel[k]; f->vel_right[k] = rec[i].vel_right[k]; }
            f->is_stereo = rec[i].is_stereo != 0;
            f->disp = (float)rec[i].disp;
            FeatureInstance& fi = out[rec[i].inst_id];
            if (fi.features.empty()) {
                auto it = instances.find(rec[i].inst_id);
                if (it != instances.end()) { fi.color = it->second.color; fi.box2d = it->second.box2d; }
            }
            fi.features.insert({rec[i].id, f});
        }
        // an instance that is visible but holds no point yet still appears in the reference's result
        for (auto& kv : instances)
            if (kv.second.lost_num == 0 && kv.second.is_curr_visible && out.count(kv.first) == 0) {
                FeatureInstance fi;
                fi.color = kv.second.color; fi.box2d = kv.second.box2d;
                out.insert({kv.first, fi});
            }
        return out;
    }

    void SetEstimatedInstancesInfo(const std::unordered_map<unsigned int, InstEstimatedInfo>& estimated_info_) {
        estimated_info = estimated_info_;
    }
    // front_end/dynamic_tracker.h:62-68
    template <class F>
    void ExecInst(F func) {
        for (auto& kv : instances) {
            if (kv.second.lost_num > 0) continue;
            func(kv.first, kv.second);
        }
    }

    std::unordered_map<unsigned int, InstFeat> instances;                    // dynamic_tracker.h:83
    std::unordered_map<unsigned int, InstEstimatedInfo> estimated_info;

private:
    static FeatureTracker* require_tracker(const std::string& config_path) {
        FeatureTracker* t = FeatureTracker::current();
        if (t == nullptr || (!t->config_path().empty() && t->config_path() != config_path))
            throw std::runtime_error("InstsFeatManager: create the FeatureTracker of this config first (the two share the "
                                     "feature-id counter and the frame on the device)");
        return t;
    }
    std::map<unsigned int, InstFeat*> sorted_instances() {
        std::map<unsigned int, InstFeat*> m;
        for (auto& kv : instances) m[kv.first] = &kv.second;
        return m;
    }
    // lost_num bookkeeping and erasure happen inside the library (ManageInstances, dynamic_tracker.cpp:499-514)
    void sync_table() {
        const int cap = t_.config().max_instances > 0 ? t_.config().max_instances : 1;
        std::vector<dvfe_inst_info> rows((size_t)cap);
        int n = 0;
        if (dvfe_insts_table(t_.handle(), 0, rows.data(), cap, &n) != DVFE_OK) throw std::runtime_error(dvfe_last_error(t_.handle()));
        std::unordered_map<unsigned int, InstFeat> kept;
        for (int i = 0; i < n; i++) {
            auto it = instances.find(rows[i].track_id);
            InstFeat f = it != instances.end() ? it->second : InstFeat();
            f.id = rows[i].track_id;
            f.lost_num = rows[i].lost_num;
            f.is_curr_visible = rows[i].is_curr_visible != 0;
            kept.insert({rows[i].track_id, f});
        }
        instances.swap(kept);
    }
    FeatureTracker& t_;
    SemanticImage prev_img_;
};

// Many cameras on one GPU: B independent FeatureTracker states advanced together, pipelined.  Not in the reference (one
// tracker configuration per process there, SURVEY §8b); this is the host-side shape of the B200 deployment: one object per
// GPU, `TrackImageAsync(frame k+1)` then `Wait()` -> results of frame k, so uploads overlap the kernels.  The images of
// stream s start at `base + s * stream_stride`.
class BatchFeatureTracker {
public:
    BatchFeatureTracker(const std::string& config_path, int n_streams, int n_groups = 4, int max_instances = 0) {
        if (dvfe_config_from_yaml(config_path.c_str(), &cfg_) != DVFE_OK) throw std::runtime_error(dvfe_last_error(nullptr));
        cfg_.n_streams = n_streams; cfg_.n_groups = n_groups; cfg_.max_instances = max_instances;
        if (dvfe_create(&cfg_, &h_) != DVFE_OK) throw std::runtime_error(dvfe_last_error(nullptr));
    }
    explicit BatchFeatureTracker(const dvfe_config& cfg) : cfg_(cfg) {
        if (dvfe_create(&cfg_, &h_) != DVFE_OK) throw std::runtime_error(dvfe_last_error(nullptr));
    }
    ~BatchFeatureTracker() { dvfe_destroy(h_); }
    BatchFeatureTracker(const BatchFeatureTracker&) = delete;
    BatchFeatureTracker& operator=(const BatchFeatureTracker&) = delete;

    int streams() const { return cfg_.n_streams; }
    const dvfe_config& config() const { return cfg_; }
    dvfe_tracker* handle() { return h_; }

    // The calibration of one stream (cam_t.cam0 / cam1 of that stream's rig, e.g. dvfe_camera_from_yaml of its calibration
    // files; cam1 == nullptr: cam1 = cam0), from the next step on; the stream's tracking state is kept (dvfe_set_stream_camera)
    void SetStreamCamera(int stream, const dvfe_camera& cam0, const dvfe_camera* cam1 = nullptr) {
        if (dvfe_set_stream_camera(h_, stream, &cam0, cam1) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
    }
    // The undistortion maps of camera `cam` for one stream (CV_16SC2 + CV_16UC1; both null: not remapped); no step may be in
    // flight (dvfe_set_stream_undistort_maps)
    void SetStreamUndistortMaps(int stream, int cam, const int16_t* map1, const uint16_t* map2) {
        if (dvfe_set_stream_undistort_maps(h_, stream, cam, map1, map2) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
    }

    // RejectWithF inside every step of every stream (dvfe_set_reject_with_f; 0 = off, the default), from the next step on
    void SetRejectWithF(double f_threshold) {
        if (dvfe_set_reject_with_f(h_, f_threshold) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
    }

    // Everything the next step of one stream reads from earlier frames, as one blob (dvfe_export_stream); no step may be in flight
    std::vector<uint8_t> ExportStream(int stream) {
        size_t n = 0;
        if (dvfe_export_stream(h_, stream, nullptr, 0, &n) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
        std::vector<uint8_t> blob(n);
        if (dvfe_export_stream(h_, stream, blob.data(), blob.size(), &n) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
        return blob;
    }
    // The whole state of slot `stream` from an exported blob (dvfe_import_stream): the slot continues as the source stream would have
    void ImportStream(int stream, const std::vector<uint8_t>& blob) {
        if (dvfe_import_stream(h_, stream, blob.data(), blob.size()) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
    }

    // TrackImage of all cameras, enqueued; `time0` has one entry per stream; the images stay valid until the matching Wait()
    void TrackImageAsync(const uint8_t* left, const uint8_t* right, size_t stream_stride, int step, const std::vector<double>& time0) {
        check(time0);
        if (dvfe_track_image_async(h_, left, right, stream_stride, step, time0.data()) != DVFE_OK)
            throw std::runtime_error(dvfe_last_error(h_));
    }
    // The same with per-stream frame presence: stream_flags[s] is 0 or DVFE_FRAME_SKIP / DVFE_FRAME_NO_RIGHT / DVFE_FRAME_RESET
    // (dvfe_track_image_ex); a skipped stream's time0 is not read.  `device`: left / right are device pointers.
    void TrackImageAsync(const uint8_t* left, const uint8_t* right, size_t stream_stride, int step, const std::vector<double>& time0,
                         const std::vector<uint8_t>& stream_flags, bool device = false) {
        check(time0);
        if ((int)stream_flags.size() != cfg_.n_streams) throw std::runtime_error("BatchFeatureTracker: one stream flag per stream expected");
        if (dvfe_track_image_ex(h_, left, right, stream_stride, step, time0.data(), stream_flags.data(),
                                device ? DVFE_STEP_DEVICE_INPUT : 0u) != DVFE_OK)
            throw std::runtime_error(dvfe_last_error(h_));
    }
    // TrackSemanticImage + InstsTrack of all cameras, enqueued (dynamic mode; FeatureTrack() in system/main.cpp:247-254)
    void TrackDynamicAsync(const uint8_t* left, const uint8_t* right, const uint8_t* inv_merge_mask, size_t stream_stride, int step,
                           const std::vector<int>& exist_inst, const std::vector<std::vector<Box2D::Ptr>>& boxes2d,
                           const std::vector<double>& time0) {
        dynamic(left, right, inv_merge_mask, stream_stride, step, exist_inst, boxes2d, time0, nullptr);
    }
    // The same with per-stream frame presence: stream_flags[s] is 0 or DVFE_FRAME_SKIP / DVFE_FRAME_NO_RIGHT / DVFE_FRAME_RESET
    // (dvfe_track_dynamic_ex2); a skipped stream has an empty box list, and its time0 and exist_inst are not read.
    void TrackDynamicAsync(const uint8_t* left, const uint8_t* right, const uint8_t* inv_merge_mask, size_t stream_stride, int step,
                           const std::vector<int>& exist_inst, const std::vector<std::vector<Box2D::Ptr>>& boxes2d,
                           const std::vector<double>& time0, const std::vector<uint8_t>& stream_flags) {
        if ((int)stream_flags.size() != cfg_.n_streams) throw std::runtime_error("BatchFeatureTracker: one stream flag per stream expected");
        dynamic(left, right, inv_merge_mask, stream_stride, step, exist_inst, boxes2d, time0, stream_flags.data());
    }
    // One step described camera by camera (dvfe_track_frames): frames[s].left == nullptr = no frame from camera s, right == nullptr
    // = left image only, each camera at its own pitch; only the present images are read.  Enqueued; the images stay valid until
    // the matching Wait().  `device`: the pointers are device memory.
    void TrackFramesAsync(const std::vector<dvfe_frame>& frames, bool device = false) {
        check_frames(frames);
        if (dvfe_track_frames(h_, frames.data(), device ? DVFE_STEP_DEVICE_INPUT : 0u) != DVFE_OK)
            throw std::runtime_error(dvfe_last_error(h_));
    }
    // TrackSemanticImage of every camera, described camera by camera (dvfe_track_semantic_frames; frames[s].mask = inv_merge_mask)
    void TrackSemanticFramesAsync(const std::vector<dvfe_frame>& frames, bool device = false) {
        check_frames(frames);
        if (dvfe_track_semantic_frames(h_, frames.data(), device ? DVFE_DYN_DEVICE_INPUT : 0u) != DVFE_OK)
            throw std::runtime_error(dvfe_last_error(h_));
    }
    // TrackSemanticImage + InstsTrack of every camera, described camera by camera (dvfe_track_dynamic_frames); a camera without a
    // frame has an empty box list.  flags: DVFE_DYN_DEVICE_INPUT | DVFE_DYN_LABELS.
    void TrackDynamicFramesAsync(const std::vector<dvfe_frame>& frames, const std::vector<std::vector<Box2D::Ptr>>& boxes2d,
                                 unsigned flags = 0u) {
        check_frames(frames);
        std::vector<dvfe_inst_in> in;
        std::vector<int> n;
        marshal(boxes2d, &in, &n);
        if (dvfe_track_dynamic_frames(h_, frames.data(), in.empty() ? nullptr : in.data(), n.data(), flags) != DVFE_OK)
            throw std::runtime_error(dvfe_last_error(h_));
    }
    // the oldest enqueued frame is finished: Features() / InstsOutput() return its results
    void Wait() {
        if (dvfe_wait(h_) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
    }
    // SetOutputFeats() of one camera (front_end/background_tracker.cpp:340-392)
    FeatureBackground Features(int stream) {
        std::vector<dvfe_obs> rec(2 * (size_t)cfg_.max_cnt);
        int n = 0;
        if (dvfe_get_features(h_, stream, rec.data(), (int)rec.size(), &n) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
        FeatureBackground fb;
        for (int i = 0; i < n; i++) {
            Vec7d v;
            for (int k = 0; k < 7; k++) v[k] = rec[i].v[k];
            fb.points[rec[i].id].emplace_back(rec[i].cam, v);
        }
        return fb;
    }
    // InstsFeatManager::Output() of one camera (front_end/dynamic_tracker.cpp:521-577)
    std::map<unsigned int, FeatureInstance> InstsOutput(int stream) {
        std::vector<dvfe_inst_obs> rec((size_t)(cfg_.max_instances > 0 ? cfg_.max_instances : 1) *
                                       (size_t)(cfg_.max_dynamic_cnt > 0 ? cfg_.max_dynamic_cnt : 1));
        int n = 0;
        if (dvfe_insts_output(h_, stream, rec.data(), (int)rec.size(), &n) != DVFE_OK) throw std::runtime_error(dvfe_last_error(h_));
        std::map<unsigned int, FeatureInstance> out;
        for (int i = 0; i < n; i++) {
            FeaturePoint::Ptr f = std::make_shared<FeaturePoint>();
            for (int k = 0; k < 3; k++) { f->point[k] = rec[i].point[k]; f->point_right[k] = rec[i].point_right[k]; }
            for (int k = 0; k < 2; k++) { f->vel[k] = rec[i].vel[k]; f->vel_right[k] = rec[i].vel_right[k]; }
            f->is_stereo = rec[i].is_stereo != 0;
            f->disp = (float)rec[i].disp;
            out[rec[i].inst_id].features.insert({rec[i].id, f});
        }
        return out;
    }

private:
    void dynamic(const uint8_t* left, const uint8_t* right, const uint8_t* inv_merge_mask, size_t stream_stride, int step,
                 const std::vector<int>& exist_inst, const std::vector<std::vector<Box2D::Ptr>>& boxes2d,
                 const std::vector<double>& time0, const uint8_t* stream_flags) {
        check(time0);
        if ((int)exist_inst.size() != cfg_.n_streams)
            throw std::runtime_error("BatchFeatureTracker: one exist_inst / box list per stream expected");
        std::vector<dvfe_inst_in> in;
        std::vector<int> n;
        marshal(boxes2d, &in, &n);
        if (dvfe_track_dynamic_ex2(h_, left, right, inv_merge_mask, stream_stride, step, exist_inst.data(),
                                   in.empty() ? nullptr : in.data(), n.data(), time0.data(), stream_flags, 0u) != DVFE_OK)
            throw std::runtime_error(dvfe_last_error(h_));
    }
    // the dvfe_inst_in array (stream by stream) and per-stream counts of a frame's box lists
    void marshal(const std::vector<std::vector<Box2D::Ptr>>& boxes2d, std::vector<dvfe_inst_in>* in, std::vector<int>* n) const {
        if ((int)boxes2d.size() != cfg_.n_streams) throw std::runtime_error("BatchFeatureTracker: one exist_inst / box list per stream expected");
        n->resize(boxes2d.size());
        for (size_t s = 0; s < boxes2d.size(); s++) {
            (*n)[s] = (int)boxes2d[s].size();
            for (const Box2D::Ptr& b : boxes2d[s]) {
                dvfe_inst_in d{};
                d.track_id = (uint32_t)b->track_id;
                d.x = (int)b->rect.x; d.y = (int)b->rect.y; d.w = (int)b->rect.width; d.h = (int)b->rect.height;
                d.mask = b->roi ? b->roi->mask_cv.data : nullptr; d.mask_pitch = b->roi ? b->roi->mask_cv.step : 0;
                in->push_back(d);
            }
        }
    }
    void check_frames(const std::vector<dvfe_frame>& frames) const {
        if ((int)frames.size() != cfg_.n_streams) throw std::runtime_error("BatchFeatureTracker: one frame descriptor per stream expected");
    }
    void check(const std::vector<double>& time0) const {
        if ((int)time0.size() != cfg_.n_streams) throw std::runtime_error("BatchFeatureTracker: one time0 per stream expected");
    }
    dvfe_config cfg_{};
    dvfe_tracker* h_ = nullptr;
};

}  // namespace dynamic_vins
