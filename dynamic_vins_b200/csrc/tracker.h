// Host-side tracker object behind the opaque `dvfe_tracker` handle of include/dvfe.h.
#pragma once
#include <map>
#include <tuple>
#include <vector>

#include "kernels.cuh"
#include "state.cuh"

struct GfttScratch {
    int n_jobs, w, h, mask_pitch, cand_cap, n_cells;
    uint8_t* mask;
    unsigned long long *cand, *cand2, *cand3;
    uint8_t* state;
    int* cell_count;
    int* counters;
};

int alloc_point_sets(PointSetArrays* S, int n_sets, int cap);
void free_point_sets(PointSetArrays* S);
int alloc_gftt_scratch(GfttScratch* sc, int n_jobs, int w, int h, float min_dist);
void free_gftt_scratch(GfttScratch* sc);
void gftt_job_bind_scratch(GfttJob* J, const GfttScratch& sc, int j);
int gftt_cells(int w, int h, float min_dist);
// Checks per-stream DVFE_FRAME_* bytes (nullable) of a tracker with B streams; *out = stream_flags, or null when no flag is set (the
// step is then the plain one).  DVFE_ERR_INVALID for unknown bits and SKIP|RESET.
int check_stream_flags(const uint8_t* stream_flags, int B, const char* who, const uint8_t** out);

struct InstanceState;   // instances.cu

// One instance of a stream snapshot (snapshot.cu, dvfe_export_stream): the host bookkeeping of InstsFeatManager::instances that the
// next frame reads.  Stored in the blob as is.
struct SnapInst {
    uint32_t track_id;
    int32_t lost_num, visible, has_box;
    int32_t x, y, w, h;                              // the box of the last frame the instance was seen in
    int32_t prev_w, prev_h;                          // size of the previous ROI crop (0: none)
};
// Where that instance's device state lives: its point set in InstanceState::pts and its previous ROI crop (dense prev_w x prev_h)
struct SnapInstDev {
    size_t set;
    uint8_t* crop;
};

// Where each stream's images of a step are: img[0] left, img[1] right, img[2] mask / label image, B entries each.  A null pointer
// is an absent image: nothing is read or copied for it.  A slab call (base + s * stride) gives a uniform table; dvfe_track_frames
// gives one entry per camera, uniform only when its cameras happen to lie in one slab.
struct StepSources {
    std::vector<ImgSrc> img[3];
    bool uniform[3] = {false, false, false};         // every stream has image c, all at one pitch, stream s at img[c][0] + s * stride[c]
    size_t stride[3] = {0, 0, 0};
    bool any(int c) const {
        for (const ImgSrc& e : img[c])
            if (e.ptr) return true;
        return false;
    }
};
// The table of a slab: every stream has each image whose base is not null
StepSources slab_sources(int B, const uint8_t* left, const uint8_t* right, const uint8_t* mask, size_t stride, int pitch,
                         size_t mask_stride, int mask_pitch);

struct dvfe_tracker;
// One step of a leaf tracker from a source table, enqueued; sflags: per-stream DVFE_FRAME_* (validated) or null.
// tracker.cu: the raw step.  instances.cu: the dynamic-mode step, whose boxes (boxes_of[s], n_boxes[s]) leaf_validate_boxes
// checked before any stream group enqueued.
int leaf_track(dvfe_tracker* t, const StepSources& src, const double* time0, const uint8_t* sflags, bool device);
int leaf_validate_boxes(dvfe_tracker* t, const dvfe_inst_in* const* boxes_of, const int* n_boxes, bool labels, const uint8_t* sflags);
int leaf_track_dynamic(dvfe_tracker* t, const StepSources& src, const int* exist_inst, const dvfe_inst_in* const* boxes_of,
                       const int* n_boxes, const double* time0, const uint8_t* sflags, unsigned flags);

// Where a frame step finds its images once dvfe_tracker::place_input has put them in place
struct StepInput {
    const uint8_t* left = nullptr;                   // device images the step copies into level 0 (null when in_place)
    const uint8_t* right = nullptr;
    size_t stride = 0;                               // bytes between the streams' images
    int pitch = 0;
    bool in_place = false;                           // level 0 of this step's pyramid slots already holds the images
    bool l0_border = false;                          // ... with its border (the gather kernel of a device table)
    bool has_right = false;
};

struct dvfe_tracker {
    // A tracker is either a leaf (owns device state for its B streams) or a container of G leaf trackers
    // ("stream groups", dvfe_config::n_groups) that splits every call by stream range.
    std::vector<dvfe_tracker*> groups;
    std::vector<int> group_first;                    // first stream of each group (size G + 1)
    dvfe_config cfg{};
    int B = 0, W = 0, H = 0, cap = 0;
    cudaStream_t st = nullptr;                       // compute stream (caller-replaceable)
    cudaStream_t cs = nullptr;                       // upload stream: H2D of step k+1 overlaps the kernels of step k
    cudaStream_t ds = nullptr;                       // download stream: D2H of step k overlaps the kernels of step k+1
    cudaStream_t rs = nullptr;                       // right-image pyramid stream: fills the SMs the selection kernel leaves idle
    bool own_stream = true;
    PyrDesc desc{};
    // Per-stream calibration (dvfe_set_stream_camera): the post kernels read d_cam[cam * B + stream].  The host table is the
    // calibration of the next step; submit() uploads it on the compute stream, ahead of that step's kernels, when it changed.
    // The device pointer never changes, so captured graphs stay valid.
    std::vector<CamParams> cams;                     // [2][B] cam0 of every stream, then cam1
    CamParams* d_cam = nullptr;                      // [2][B]
    CamParams* h_cam[2] = {nullptr, nullptr};        // pinned copy source, one per in-flight step
    bool cam_dirty = false;                          // `cams` differs from what the last uploaded table holds
    // Pyramids: 3 left slots (current / previous / being uploaded) and 2 right slots.  Step k uses
    // left[k % 3] (previous = left[(k + 2) % 3]) and right[k % 2]; "phase" = k % 6 selects the descriptor set.
    uint8_t* pyrL[3] = {nullptr, nullptr, nullptr};
    uint8_t* pyrR[2] = {nullptr, nullptr};
    long frames = 0;                                 // steps submitted
    long completed = 0;                              // steps whose outputs have been waited for
    bool last_has_right = false;                     // the last submitted frame had a right image
    std::vector<uint8_t> last_sflags;                // [B] DVFE_FRAME_* of the last submitted step (all 0 for a full step): the
                                                     // InstsTrack of the same frame follows them
    std::vector<uint8_t> had_frame;                  // [B] the stream has had a frame: the previous left slot holds its last image
    // dvfe_import_stream put a previous left image into a tracker that has run no step: its first step is then run in the
    // "not the first frame" form (temporal LK + compaction), which is exact for every stream that never had a frame (n = 0)
    bool prev_loaded = false;
    uint8_t* d_snap = nullptr;                       // stream snapshot staging (snapshot.cu), allocated on first use at its largest
    PointSetArrays bg{};                             // background point sets, one per stream
    uint32_t* d_next_id = nullptr;                   // [B] InstFeat::global_id_count per stream
    double* d_dt = nullptr;
    double* h_dt[2] = {nullptr, nullptr};
    std::vector<double> prev_time;
    dvfe_obs* d_obs[2] = {nullptr, nullptr};         // one per in-flight step
    dvfe_obs* h_obs[2] = {nullptr, nullptr};         // pinned, one per in-flight step
    int* d_nobs[2] = {nullptr, nullptr};
    int* h_nobs[2] = {nullptr, nullptr};             // [B + 1]: counts, then the device error word of that step
    int* d_err = nullptr;                            // [2]: one capacity-overflow flag per in-flight step
    int out_slot = 0;                                // which h_obs holds the newest completed step
    cudaEvent_t ev_up[2] = {}, ev_packed[2] = {}, ev_done[2] = {}, ev_resp[2] = {}, ev_rpyr[2] = {}, ev_r0[2] = {}, ev_begin[2] = {};
    uint8_t *d_region = nullptr, *d_region_tmp = nullptr;
    uint8_t* d_inv_in[2] = {nullptr, nullptr};       // uploaded inv_merge_mask, one per in-flight step
    int* d_exist = nullptr;
    int* h_exist[2] = {nullptr, nullptr};            // pinned, one per in-flight step
    cudaEvent_t ev_inst[2] = {};                     // instance records of the step are on the host
    bool inst_pending[2] = {false, false};           // the step carried a deferred InstsTrack (dvfe_track_dynamic_async)
    GfttScratch gsc{};
    LkGroup* d_groups[6][3] = {};                    // [phase][temporal raw | temporal semantic | stereo]
    GfttJob* d_jobs[6][3] = {};                      // [phase][raw | semantic | semantic, cv::cuda detector threshold]
    InstanceState* inst = nullptr;
    unsigned* d_tcache = nullptr;                    // LK template cache [B][cap][DVFE_MAX_PYR_LEVELS][LK_TCACHE_WORDS] (stereo only)
    bool tcache_valid = false;                       // the last step ran the stereo LK on the points `bg` holds now
    unsigned* d_tcache_bwd = nullptr;                // backward templates of the temporal call, same layout (stereo only)
    int* d_old_idx = nullptr;                        // [B][cap] index of each point in the temporal call of the step, -1 = new
    // Per-stream frame presence (dvfe_track_image_ex).  A "partial" step (any stream flag set) runs the same kernels on tables
    // rebuilt from the stream flags at its start; steps without flags never touch any of this.
    uint8_t* h_sflags[2] = {nullptr, nullptr};       // pinned [B] per in-flight step: DVFE_FRAME_* | SF_TCACHE_VALID
    uint8_t* d_sflags = nullptr;                     // [B] the flags of the step on the compute stream
    uint8_t* d_lane = nullptr;                       // [B] 0 = skipped, else LANE_PRESENT | LANE_STEREO (compact, left/right post)
    LkGroup* d_pgroups[2] = {nullptr, nullptr};      // [B] partial temporal / stereo LK tables
    GfttJob* d_pjobs = nullptr;                      // [B] partial GFTT jobs
    int* d_zero = nullptr;                           // the point count of a stream an LK table leaves out
    std::vector<uint8_t> tc_valid;                   // per stream: d_tcache holds the forward templates of its current points
    // backward LK maxLevel / forward-backward threshold per call site [DVFE_LK_*]: the CPU FeatureTrackByLK pair
    // (feature_utils.cpp:51,57: 1, 0.5) everywhere except TrackSemanticImage's right image, which the reference tracks with
    // the cv::cuda call pattern (TrackRightGPU, background_tracker.cpp:801: 3 levels, 1.0 px)
    int lk_back_level[4] = {1, 1, 1, 3};
    double lk_fb_thresh[4] = {0.5, 0.5, 0.5, 1.0};
    // dvfe_set_reject_with_f: F_threshold of the in-step RejectWithF (0 = off) and the model scratch of its kernel (allocated when
    // first enabled)
    double reject_f = 0.0;
    double* d_fm_models = nullptr;

    // The compute part of a frame step is a fixed launch sequence for a given buffer phase, input location and mode: it is
    // captured once into a CUDA graph and replayed (one launch per step and stream group instead of ~20).
    typedef std::tuple<int, unsigned> StepKey;       // buffer phase, mode flags (the caller's image pointers stay outside)
    struct StepGraph { cudaGraphExec_t exec = nullptr; unsigned n_kernels = 0; };
    std::map<StepKey, StepGraph> step_graphs;
    bool detect_cuda = false;                        // dvfe_set_detect_mode: semantic-path detection with the cv::cuda detector's threshold
    bool use_graphs = true;
    bool use_reuse = true;                           // DVFE_REUSE=0: the stereo call rebuilds every forward template (A/B, debugging)
    void drop_graphs();
    int capture_step(int ph, unsigned flags, long k);
    int enqueue_compute(const uint8_t* d_left, const uint8_t* d_right, size_t stream_stride, int pitch, bool semantic,
                        int level0_mode, bool stereo_now, long k, bool with_marks, bool partial = false);

    // per-stage device timers (one event set per in-flight step)
    enum { ST_PYRAMID, ST_LK_TEMPORAL, ST_COMPACT, ST_GFTT_MASK, ST_GFTT_DISCS, ST_GFTT_RESPONSE, ST_GFTT_SELECT, ST_LEFT_POST,
           ST_LK_STEREO, ST_PACK, ST_D2H, ST_COUNT };
    bool prof = false;
    bool prof_step[2] = {false, false};
    cudaEvent_t ev[2][ST_COUNT + 1] = {};
    double prof_ms[ST_COUNT] = {};
    long prof_steps = 0;

    // TMA descriptors (CUtensorMap, 128 B each) over level 0 of the three left pyramid sets: the corner response loads its
    // tiles with cp.async.bulk.tensor; use_tma is false when the driver cannot encode them (then cp.async is used)
    alignas(64) unsigned char tmapL[3][128] = {};
    bool use_tma = false;
    uint8_t* left_slot(long k) const { return pyrL[k % 3]; }
    uint8_t* right_slot(long k) const { return pyrR[k % 2]; }

    int init();
    int init_instances();
    void free_instances();
    bool staged_upload = false;                      // rows that are not a multiple of 64 B make pitched DMA slow
    // frame ingest (dvfe_set_input / dvfe_set_undistort_maps): BGR and/or remapped input goes through a device staging
    // buffer and the ingest kernel, which writes level 0 in place
    int in_ch = 1;
    short* d_map1[2] = {nullptr, nullptr};           // the maps of every stream of camera cam (dvfe_set_undistort_maps)
    unsigned short* d_map2[2] = {nullptr, nullptr};
    // per-stream maps (dvfe_set_stream_undistort_maps): own_maps[cam][s] = the stream's own maps (or none) replace the shared ones
    std::vector<uint8_t> own_maps[2];
    std::vector<short*> s_map1[2];                   // [B], null = no maps
    std::vector<unsigned short*> s_map2[2];
    IngestMaps* d_imaps[2] = {nullptr, nullptr};     // [B] the maps each image of camera cam is remapped with (ingest kernel)
    bool maps_uniform[2] = {true, true};             // every stream of camera cam uses the same maps: the shared-map kernel
    const short* stream_map1(int cam, int s) const { return own_maps[cam][s] ? s_map1[cam][s] : d_map1[cam]; }
    const unsigned short* stream_map2(int cam, int s) const { return own_maps[cam][s] ? s_map2[cam][s] : d_map2[cam]; }
    int update_maps(int cam);                        // recompute maps_uniform[cam] and upload d_imaps[cam] (no step in flight)
    // dense staging of host images [2 cameras][B][H*W*in_ch], one per in-flight step: the staged upload's copy source, or the
    // ingest kernel's input; sized by size_stage() whenever the input format changes, never inside a step
    uint8_t* d_stage[2] = {nullptr, nullptr};
    bool prep_active() const {                       // any stream of either camera has maps, or BGR input
        if (in_ch != 1) return true;
        for (int cam = 0; cam < 2; cam++)
            for (int s = 0; s < B; s++)
                if (stream_map1(cam, s)) return true;
        return false;
    }
    int size_stage();
    uint8_t* level0(int cam) const;                  // the interior of level 0 of this step's left / right slot
    int ingest(const uint8_t* d_src, size_t stream_stride, int pitch, int cam, cudaStream_t s);
    int h2d(uint8_t* dst, size_t dst_pitch, size_t dst_stride, const uint8_t* src, size_t src_pitch, size_t src_stride, size_t row);
    int wait_slot();                                 // fewer than two steps in flight: step k-2's buffers are free again
    // wait_slot, then put this step's images (host or device memory) where the step reads them
    int place_input(const StepSources& src, bool device, StepInput* in);
    int place_table(const StepSources& src, bool device, StepInput* in);     // the routes of a table that is not uniform
    // the slab table of this tracker: the mask / label image is one byte per pixel at the stride and pitch of the images divided
    // by the channel count when the ingest kernel runs
    StepSources slab(const uint8_t* left, const uint8_t* right, const uint8_t* mask, size_t stride, int pitch) const;
    // Per-step device copy of a table's pointers ([3][B], for the gather kernels), uploaded on the compute stream from a pinned
    // copy per in-flight step; read only by kernels on the compute stream, so one device table serves every step
    ImgSrc* d_src = nullptr;
    ImgSrc* h_src[2] = {nullptr, nullptr};
    long src_step = -1;                              // the step whose table d_src holds
    int upload_sources(const StepSources& src);
    // enqueue one frame step (no host synchronisation); at most two steps are in flight
    // sflags (nullable): per-stream DVFE_FRAME_* (dvfe_track_image_ex / _semantic_ex / _dynamic_ex2), already validated
    int submit(const StepInput& in, const double* time0, bool semantic, const uint8_t* sflags = nullptr);
    // TrackSemanticImage of one frame, enqueued only (uploads on the copy stream, mask erosion + the frame step)
    // flags: DVFE_DYN_DEVICE_INPUT (the three pointers are device memory, nothing is uploaded), DVFE_DYN_LABELS (the mask is a
    // label image: the region is everything no instance bit is set on).  sflags: as submit; a skipped stream's exist_inst and
    // mask are not read, a RESET stream's instance manager starts over too
    int semantic_submit(const StepSources& src, const int* exist_inst, const double* time0, unsigned flags = 0,
                        const uint8_t* sflags = nullptr);
    void reset_instances(int stream);                // instances.cu: a newly created InstsFeatManager for one stream
    // instances.cu, for stream snapshots: the instance table of `stream` in ascending track id with where each instance's device state
    // lives, and its last_time; insts_import replaces the table (slots from the free list) and says where the device state goes
    void insts_export(int stream, std::vector<SnapInst>* recs, std::vector<SnapInstDev>* dev, double* last_time) const;
    void insts_import(int stream, const std::vector<SnapInst>& recs, double last_time, std::vector<SnapInstDev>* dev);
    const PointSetArrays& inst_points() const;
    uint8_t* d_labels[2] = {nullptr, nullptr};       // uploaded label images, one per in-flight step (allocated on first use)
    const uint8_t* lab_ptr[2] = {nullptr, nullptr};  // the label images of the in-flight steps (device), for the ROI masks
    size_t lab_stride[2] = {0, 0};
    int lab_pitch[2] = {0, 0};
    int finish_instances(int par);                   // instances.cu: host side of a deferred InstsTrack
    int wait_one();                                  // oldest in-flight step -> outputs readable
    int wait_all();
};
