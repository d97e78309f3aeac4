// Per-instance tracking — replaces InstsFeatManager::InstsTrack / ManageInstances / Output / AddViodeInstances
// (dynamic_vins/src/front_end/dynamic_tracker.cpp:348-493, 499-514, 521-577, 585-605) and the caller's per-frame
// instance reset (dynamic_vins/src/system/main.cpp:198-202), minus the DeepSORT / PCL / 3-D box branches.
//
// Host side: the instance table (track id -> slot, lost_num, visibility, boxes) — the same bookkeeping the
// reference does on the host.  Device side: every visible instance of the frame is one job of each batched
// launch (ROI crop, zero-padded ROI pyramids, LK on the previous-box crop -> current-box crop in ROI-local
// coordinates, mask erosion, Shi-Tomasi on the ROI, offset undistortion, full-image left->right LK).
//
// Order of feature-id assignment: the background step of the frame (dvfe_track_semantic_image) runs first, then
// the instances in ascending instance id (the reference races the two threads on one counter and iterates an
// unordered_map; see oracle/cv_front_end.py header).
#include <math.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <vector>

#include "kernels.cuh"
#include "state.cuh"
#include "tracker.h"

#define DVFE_CHECK(call)                 \
    do {                                 \
        int rc__ = (call);               \
        if (rc__ != DVFE_OK) return rc__; \
    } while (0)

namespace {
struct InstHost {
    uint32_t track_id = 0;
    int slot = -1;
    int lost_num = 0;
    bool visible = false;          // is_curr_visible
    bool has_box = false;          // box2d != nullptr
    int x = 0, y = 0, w = 0, h = 0;      // box2d->rect of the current frame
    int prev_w = 0, prev_h = 0;    // size of roi->prev_roi_gray (0 = empty)
    int cur_buf = 0;               // which of the two ROI buffers holds roi_gray
    int roi_w = 0, roi_h = 0;      // size of roi->roi_gray
    long long mask_off = -1;       // offset of this frame's ROI mask in the packed staging (-1: in the slot buffer)
    int label_bit = -1;            // >= 0: the ROI mask is bit `label_bit` of the frame's label image (device)
    const float* disp = nullptr;   // SemanticImage::disp of this frame (host, full image size) or null
    int disp_pitch = 0;
};

struct InstStream {
    std::map<uint32_t, InstHost> insts;      // ascending instance id = the deterministic ExecInst order
    std::vector<int> free_slots;
    double last_time = 0.0;
    std::vector<dvfe_inst_obs> out;          // Output() of the last call
};

template <typename T>
int dmalloc(T** p, size_t count) {
    DVFE_CUDA(cudaMalloc((void**)p, count * sizeof(T)));
    DVFE_CUDA(cudaMemset(*p, 0, count * sizeof(T)));
    return DVFE_OK;
}

// a per-call descriptor array: a view into the tracker's descriptor arena (one pinned blob, one device blob, ONE
// host-to-device copy per call)
template <typename T>
struct Staged {
    T* h = nullptr;
    T* d = nullptr;
};

struct Arena {
    uint8_t* h = nullptr;
    uint8_t* d = nullptr;
    size_t cap = 0, used = 0;
    int alloc(size_t bytes) {
        cap = bytes;
        DVFE_CUDA(cudaMallocHost((void**)&h, bytes));
        DVFE_CUDA(cudaMalloc((void**)&d, bytes));
        return DVFE_OK;
    }
    template <typename T>
    void take(Staged<T>& s, int n) {
        used = (used + 15) & ~(size_t)15;
        s.h = reinterpret_cast<T*>(h + used);
        s.d = reinterpret_cast<T*>(d + used);
        used += sizeof(T) * (size_t)n;
    }
    int push(cudaStream_t st) {
        DVFE_CUDA(cudaMemcpyAsync(d, h, used, cudaMemcpyHostToDevice, st));
        return DVFE_OK;
    }
    void release() {
        if (h) cudaFreeHost(h);
        if (d) cudaFree(d);
        h = d = nullptr;
    }
};
}  // namespace

// Everything one InstsTrack call hands to the device and gets back: descriptor arena, packed ROI masks, output records.
// Two of them, indexed by the parity of the frame step the call belongs to, so that a deferred call
// (dvfe_track_dynamic_async) can be prepared while the previous step is still running.
struct InstCall {
    Arena arena;                         // per-call descriptors (NS entries each), one pinned blob + one device blob
    uint8_t *h_mask_stage = nullptr, *d_mask_stage = nullptr;    // packed ROI masks of one call (pinned / device)
    Staged<CropJob> crop;
    Staged<PyrJob> pyr;                  // 2*NS
    Staged<LkGroup> lk_t, lk_s;
    Staged<ErodeJob> erode;
    Staged<GfttJob> gftt;
    Staged<uint8_t> act_track, act_vis, clear_flags;    // indexed by set
    Staged<uint8_t> lane;                // per set, after a step with stream flags: LANE_PRESENT | LANE_STEREO of its stream
    Staged<double> dt;
    Staged<float2> offs;
    Staged<uint32_t> inst_id;
    dvfe_inst_obs* d_out = nullptr;      // [NS*cap]
    dvfe_inst_obs* h_out = nullptr;      // pinned
    int* d_n = nullptr;                  // [NS] record counts of THIS call (snapshot of the point-set counts)
    int* h_n = nullptr;                  // pinned [NS + 1]: counts, then the step's capacity-overflow word after the ROI detections
    cudaEvent_t ev_packed = nullptr;     // instance kernels of the call are done (compute stream)
    cudaEvent_t ev_up = nullptr;         // masks + descriptors of the call are on the device (upload stream)
    // host side of Output(), fixed when the call is enqueued
    int s0 = 0, s1 = 0;                  // streams whose Output() this call replaces
    struct Planned { int stream, set; const float* disp; int disp_pitch; };
    std::vector<Planned> plan;           // the visible instances in output order (+ the disparity map Output() reads)
    bool has_records = false;            // the call launched kernels (h_n / h_out are meaningful)
};

struct InstanceState {
    int MI = 0, cap = 0;                 // slots per stream, points per slot (max_dynamic_cnt)
    size_t P = 0;                        // W*H: capacity of one ROI buffer
    PyrDesc full{};                      // capacity of one ROI pyramid
    std::vector<InstStream> streams;
    PointSetArrays pts{};                // B*MI sets
    uint8_t *roi_gray = nullptr;         // [B*MI][2][P]
    uint8_t *roi_mask = nullptr, *roi_mask_tmp = nullptr, *roi_mask_er = nullptr;   // [B*MI][P]
    uint8_t *pyr_prev = nullptr, *pyr_cur = nullptr;                                 // [B*MI][full.bytes]
    GfttScratch gsc{};                   // B*MI jobs at full image size
    size_t mask_stage_cap = 0;
    InstCall call[2];
};

int dvfe_tracker::init_instances() {
    if (cfg.max_instances <= 0) return DVFE_OK;
    if (cfg.max_dynamic_cnt < 1 || cfg.max_dynamic_cnt > 2048 || cfg.min_dynamic_dist < 1) {
        dvfe_set_error("dvfe_create: invalid instance config (max_dynamic_cnt=%d min_dynamic_dist=%d)", cfg.max_dynamic_cnt,
                       cfg.min_dynamic_dist);
        return DVFE_ERR_CONFIG;
    }
    inst = new InstanceState();
    InstanceState& I = *inst;
    I.MI = cfg.max_instances; I.cap = cfg.max_dynamic_cnt; I.P = (size_t)W * H;
    I.full = make_pyr_desc(W, H, cfg.lk_max_level > 3 ? cfg.lk_max_level : 3);
    const size_t NS = (size_t)B * I.MI;
    I.streams.resize(B);
    for (int s = 0; s < B; s++) reset_instances(s);
    DVFE_CHECK(alloc_point_sets(&I.pts, (int)NS, I.cap));
    DVFE_CHECK(dmalloc(&I.roi_gray, NS * 2 * I.P));
    DVFE_CHECK(dmalloc(&I.roi_mask, NS * I.P));
    DVFE_CHECK(dmalloc(&I.roi_mask_tmp, NS * I.P));
    DVFE_CHECK(dmalloc(&I.roi_mask_er, NS * I.P));
    DVFE_CHECK(dmalloc(&I.pyr_prev, NS * I.full.bytes));
    DVFE_CHECK(dmalloc(&I.pyr_cur, NS * I.full.bytes));
    DVFE_CHECK(alloc_gftt_scratch(&I.gsc, (int)NS, W, H, (float)cfg.min_dynamic_dist));
    I.mask_stage_cap = (size_t)(B < 4 ? 4 : B) * I.P;      // ROI masks of one call, packed
    for (int p = 0; p < 2; p++) {
        InstCall& C = I.call[p];
        DVFE_CHECK(dmalloc(&C.d_out, NS * I.cap));
        DVFE_CHECK(dmalloc(&C.d_n, NS));
        DVFE_CUDA(cudaMallocHost((void**)&C.h_out, NS * I.cap * sizeof(dvfe_inst_obs)));
        DVFE_CUDA(cudaMallocHost((void**)&C.h_n, (NS + 1) * sizeof(int)));
        memset(C.h_n, 0, (NS + 1) * sizeof(int));
        DVFE_CHECK(C.arena.alloc(NS * (sizeof(CropJob) + 2 * sizeof(PyrJob) + 2 * sizeof(LkGroup) + sizeof(ErodeJob) +
                                       sizeof(GfttJob) + 4 + sizeof(double) + sizeof(float2) + sizeof(uint32_t)) + 4096));
        C.arena.take(C.crop, (int)NS);
        C.arena.take(C.pyr, 2 * (int)NS);
        C.arena.take(C.lk_t, (int)NS);
        C.arena.take(C.lk_s, (int)NS);
        C.arena.take(C.erode, (int)NS);
        C.arena.take(C.gftt, (int)NS);
        C.arena.take(C.act_track, (int)NS);
        C.arena.take(C.act_vis, (int)NS);
        C.arena.take(C.clear_flags, (int)NS);
        C.arena.take(C.lane, (int)NS);
        C.arena.take(C.dt, (int)NS);
        C.arena.take(C.offs, (int)NS);
        C.arena.take(C.inst_id, (int)NS);
        DVFE_CUDA(cudaMallocHost((void**)&C.h_mask_stage, I.mask_stage_cap));
        DVFE_CHECK(dmalloc(&C.d_mask_stage, I.mask_stage_cap));
        DVFE_CUDA(cudaEventCreateWithFlags(&C.ev_packed, cudaEventDisableTiming));
        DVFE_CUDA(cudaEventCreateWithFlags(&C.ev_up, cudaEventDisableTiming));
    }
    return DVFE_OK;
}

void dvfe_tracker::free_instances() {
    if (!inst) return;
    InstanceState& I = *inst;
    free_point_sets(&I.pts);
    cudaFree(I.roi_gray); cudaFree(I.roi_mask); cudaFree(I.roi_mask_tmp); cudaFree(I.roi_mask_er);
    cudaFree(I.pyr_prev); cudaFree(I.pyr_cur);
    free_gftt_scratch(&I.gsc);
    for (int p = 0; p < 2; p++) {
        InstCall& C = I.call[p];
        cudaFree(C.d_out); cudaFree(C.d_n); cudaFreeHost(C.h_out); cudaFreeHost(C.h_n);
        C.arena.release();
        if (C.h_mask_stage) cudaFreeHost(C.h_mask_stage);
        cudaFree(C.d_mask_stage);
        if (C.ev_packed) cudaEventDestroy(C.ev_packed);
        if (C.ev_up) cudaEventDestroy(C.ev_up);
    }
    delete inst;
    inst = nullptr;
}

// a newly created InstsFeatManager for `stream` (DVFE_FRAME_RESET): no instances, every slot free, last_time = 0.  A slot's
// point count is cleared when an instance takes it; Output() of the last completed call stays readable.
void dvfe_tracker::reset_instances(int stream) {
    InstStream& S = inst->streams[stream];
    S.insts.clear();
    S.free_slots.clear();
    for (int k = inst->MI - 1; k >= 0; k--) S.free_slots.push_back(k);
    S.last_time = 0.0;
}

// The previous ROI crop of an instance is in the buffer its last crop went to (cur_buf); an imported one goes to buffer 0.
void dvfe_tracker::insts_export(int stream, std::vector<SnapInst>* recs, std::vector<SnapInstDev>* dev, double* last_time) const {
    const InstStream& S = inst->streams[stream];
    for (const auto& kv : S.insts) {
        const InstHost& in = kv.second;
        recs->push_back(SnapInst{in.track_id, in.lost_num, in.visible ? 1 : 0, in.has_box ? 1 : 0, in.x, in.y, in.w, in.h,
                                 in.prev_w, in.prev_h});
        const size_t set = (size_t)stream * inst->MI + in.slot;
        dev->push_back(SnapInstDev{set, inst->roi_gray + (set * 2 + in.cur_buf) * inst->P});
    }
    *last_time = S.last_time;
}

void dvfe_tracker::insts_import(int stream, const std::vector<SnapInst>& recs, double last_time, std::vector<SnapInstDev>* dev) {
    reset_instances(stream);
    InstStream& S = inst->streams[stream];
    S.last_time = last_time;
    S.out.clear();
    for (const SnapInst& r : recs) {
        InstHost in;
        in.track_id = r.track_id;
        in.slot = S.free_slots.back();
        S.free_slots.pop_back();
        in.lost_num = r.lost_num; in.visible = r.visible != 0; in.has_box = r.has_box != 0;
        in.x = r.x; in.y = r.y; in.w = r.w; in.h = r.h;
        in.prev_w = r.prev_w; in.prev_h = r.prev_h;
        in.roi_w = r.prev_w; in.roi_h = r.prev_h;
        in.cur_buf = 0;
        S.insts.emplace(r.track_id, in);
        const size_t set = (size_t)stream * inst->MI + in.slot;
        dev->push_back(SnapInstDev{set, inst->roi_gray + set * 2 * inst->P});
    }
}

const PointSetArrays& dvfe_tracker::inst_points() const { return inst->pts; }

// InstsFeatManager::ManageInstances (front_end/dynamic_tracker.cpp:499-514)
static void manage_instances(InstStream& S) {
    for (auto it = S.insts.begin(); it != S.insts.end();) {
        InstHost& in = it->second;
        if (in.lost_num == 0 && !in.has_box) in.lost_num++;
        if (in.lost_num > 0) {
            in.lost_num++;
            if (in.lost_num > 3) {
                S.free_slots.push_back(in.slot);
                it = S.insts.erase(it);
                continue;
            }
        }
        ++it;
    }
}

// Every box inside the image with a mask, no box for a skipped stream, and enough free slots for the new track ids: checked before
// anything is changed (and, for the pipelined call, before the background step is enqueued), so a bad call leaves the tracker
// untouched.  sflags (nullable, [B]): the stream flags of the frame; a RESET stream's instance table counts as empty.
static int insts_validate(dvfe_tracker* t, int s0, int s1, const dvfe_inst_in* const* boxes_of, const int* n_of, bool labels,
                          const uint8_t* sflags) {
    InstanceState& I = *t->inst;
    const int W = t->W, H = t->H;
    for (int stream = s0; stream < s1; stream++) {
        const InstStream& S = I.streams[stream];
        const dvfe_inst_in* boxes = boxes_of[stream - s0];
        const unsigned sf = sflags ? sflags[stream] : 0u;
        if ((sf & DVFE_FRAME_SKIP) && n_of[stream - s0] > 0) {
            dvfe_set_error("insts_track: stream %d skips this frame but has %d boxes", stream, n_of[stream - s0]);
            return DVFE_ERR_INVALID;
        }
        const bool fresh_table = (sf & DVFE_FRAME_RESET) != 0;
        std::vector<uint32_t> fresh;
        for (int b = 0; b < n_of[stream - s0]; b++) {
            const dvfe_inst_in& bx = boxes[b];
            const bool mask_ok = labels ? (bx.label_bit >= 0 && bx.label_bit < 8) : (bx.mask != nullptr && bx.mask_pitch >= bx.w);
            if (bx.w < 1 || bx.h < 1 || bx.x < 0 || bx.y < 0 || bx.x + bx.w > W || bx.y + bx.h > H || !mask_ok ||
                (bx.disp != nullptr && bx.disp_pitch < (int)(W * sizeof(float)))) {
                dvfe_set_error("insts_track: stream %d box %d (%d,%d,%d,%d) is outside the %dx%d image or has no mask / label bit",
                               stream, b, bx.x, bx.y, bx.w, bx.h, W, H);
                return DVFE_ERR_INVALID;
            }
            if ((fresh_table || S.insts.find(bx.track_id) == S.insts.end()) &&
                std::find(fresh.begin(), fresh.end(), bx.track_id) == fresh.end())
                fresh.push_back(bx.track_id);
        }
        if (fresh.size() > (fresh_table ? (size_t)I.MI : S.free_slots.size())) {
            dvfe_set_error("insts_track: more than max_instances=%d live instances in stream %d", I.MI, stream);
            return DVFE_ERR_CAPACITY;
        }
    }
    return DVFE_OK;
}

// InstsTrack for the streams [s0, s1): boxes_of[s - s0] / n_of[s - s0] / time_of[s - s0].  Every visible instance of
// every stream is one job of each batched launch; one descriptor upload, one mask upload, one synchronisation.
// defer = false: synchronous (the background step has been waited for; ends with a synchronisation and Output() ready).
// defer = true: enqueue only, behind the background step just submitted; the records come home on the download stream and
// dvfe_tracker::wait_one() finishes the call (finish_instances).  Nothing on the host side depends on device results.
// labels: the ROI masks are cut out of the label images the background step of this frame received (DVFE_DYN_LABELS) on the
// device, inside the erosion that reads them; no mask bytes cross the bus.
// The stream flags of the last background step apply: a skipped stream is not touched (no per-frame reset, no lost_num change,
// no ManageInstances, last_time kept), a NO_RIGHT stream runs mono, a RESET stream's table was cleared by that step.
static int insts_track_streams(dvfe_tracker* t, int s0, int s1, const dvfe_inst_in* const* boxes_of, const int* n_of,
                               const double* time_of, bool defer, bool labels = false) {
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    const uint8_t* sflags = t->last_sflags.data();
    // deferred: validated before the background step
    if (!defer) DVFE_CHECK(insts_validate(t, s0, s1, boxes_of, n_of, labels, sflags));
    if (!defer) DVFE_CHECK(t->wait_all());
    InstanceState& I = *t->inst;
    const int par = (int)((t->frames - 1) % 2);          // the step these instances belong to
    InstCall& C = I.call[par];
    cudaStream_t st = t->st;
    const int W = t->W, H = t->H, MI = I.MI, cap = I.cap, B = t->B;
    const size_t P = I.P;
    const int NS = B * MI;
    // the frame uploaded by the last background step
    const PyrLevel& L0 = t->desc.lv[0];
    const bool stereo_now = t->cfg.stereo && t->last_has_right;
    bool partial = false;
    for (int stream = s0; stream < s1; stream++) partial = partial || sflags[stream] != 0;

    memset(C.act_track.h, 0, NS); memset(C.act_vis.h, 0, NS); memset(C.clear_flags.h, 0, NS);
    size_t mask_used = 0;
    int nv = 0, n_track = 0, n_stereo = 0, max_rw = 1, max_rh = 1, max_pw = 1, max_ph = 1, max_lv = 1;
    bool any_clear = false;
    std::vector<char> exist(s1 - s0, 0);
    C.s0 = s0; C.s1 = s1; C.plan.clear(); C.has_records = false;
    C.h_n[NS] = 0;

    for (int stream = s0; stream < s1; stream++) {
        if (sflags[stream] & DVFE_FRAME_SKIP) continue;                  // InstsTrack is not called for this stream
        const bool stereo = stereo_now && !(sflags[stream] & DVFE_FRAME_NO_RIGHT);
        InstStream& S = I.streams[stream];
        const dvfe_inst_in* boxes = boxes_of[stream - s0];
        const int n_boxes = n_of[stream - s0];
        const double time0 = time_of[stream - s0];
        const size_t base_set = (size_t)stream * MI;
        const uint8_t* left_pyr = t->left_slot(t->frames - 1) + (size_t)stream * t->desc.bytes;
        const uint8_t* right_pyr = t->right_slot(t->frames - 1) + (size_t)stream * t->desc.bytes;
        const uint8_t* left_px = left_pyr + L0.offset + (size_t)DVFE_PADY * L0.pitch + DVFE_PADX;

        // ---- caller's per-frame reset (system/main.cpp:198-202) + AddViodeInstances (dynamic_tracker.cpp:585-605) ----
        for (auto& kv : S.insts) { kv.second.visible = false; kv.second.has_box = false; }
        for (int b = 0; b < n_boxes; b++) {
            const dvfe_inst_in& bx = boxes[b];
            auto it = S.insts.find(bx.track_id);
            if (it == S.insts.end()) {
                InstHost in;                               // a free slot exists: insts_validate
                in.track_id = bx.track_id;
                in.slot = S.free_slots.back();
                S.free_slots.pop_back();
                DVFE_CUDA(cudaMemsetAsync(I.pts.n + base_set + in.slot, 0, sizeof(int), st));
                it = S.insts.emplace(bx.track_id, in).first;
            }
            InstHost& in = it->second;
            in.x = bx.x; in.y = bx.y; in.w = bx.w; in.h = bx.h;
            in.visible = true; in.has_box = true;
            in.disp = bx.disp; in.disp_pitch = bx.disp_pitch;
            in.label_bit = labels ? bx.label_bit : -1;
            if (labels) { in.mask_off = -1; continue; }
            // inst.roi->mask_cv = det_box->roi->mask_cv : packed into the pinned staging, uploaded with one copy below
            const size_t bytes = (size_t)bx.w * bx.h;
            if (mask_used + bytes <= I.mask_stage_cap) {
                for (int r = 0; r < bx.h; r++)
                    memcpy(C.h_mask_stage + mask_used + (size_t)r * bx.w, bx.mask + (size_t)r * bx.mask_pitch, bx.w);
                in.mask_off = (long long)mask_used;
                mask_used += (bytes + 15) & ~(size_t)15;
            } else {
                in.mask_off = -1;      // does not fit the staging area: direct (pageable) copy into the slot buffer
                DVFE_CUDA(cudaMemcpy2DAsync(I.roi_mask + (base_set + in.slot) * P, bx.w, bx.mask, bx.mask_pitch, bx.w, bx.h,
                                            cudaMemcpyHostToDevice, st));
            }
        }
        // ---- lost_num bookkeeping (:355-362) ----
        for (auto& kv : S.insts) {
            if (!kv.second.visible) kv.second.lost_num++;
            else kv.second.lost_num = 0;
        }
        exist[stream - s0] = n_boxes > 0;
        if (!exist[stream - s0]) {
            manage_instances(S);
            // ClearState (:41-58) for the instances ExecInst still visits (lost_num == 0)
            for (auto& kv : S.insts)
                if (kv.second.lost_num == 0) { C.clear_flags.h[base_set + kv.second.slot] = 1; any_clear = true; }
            S.last_time = time0;
            continue;
        }
        // jobs in ascending instance id; every job is a visible instance (lost_num == 0)
        for (auto& kv : S.insts) {
            InstHost& in = kv.second;
            if (in.lost_num != 0) continue;
            const size_t set = base_set + in.slot;
            const int j = nv++;
            // roi_gray = gray0(rect): crop into the buffer that does not hold prev_roi_gray
            in.cur_buf = in.prev_w > 0 ? 1 - in.cur_buf : in.cur_buf;
            in.roi_w = in.w; in.roi_h = in.h;
            CropJob& c = C.crop.h[j];
            c.src = left_px; c.spitch = L0.pitch; c.x = in.x; c.y = in.y; c.w = in.w; c.h = in.h;
            c.dst = I.roi_gray + (set * 2 + in.cur_buf) * P;
            max_rw = std::max(max_rw, in.w); max_rh = std::max(max_rh, in.h);
            C.act_vis.h[set] = 1;
            C.lane.h[set] = (uint8_t)(LANE_PRESENT | (stereo ? LANE_STEREO : 0u));
            C.dt.h[set] = time0 - S.last_time;                         // curr_time - last_time
            C.offs.h[set] = make_float2((float)in.x, (float)in.y);       // box2d->rect.tl()
            C.inst_id.h[set] = in.track_id;
            if (in.prev_w > 0) {
                // InstanceImagePadding: both crops zero-padded to (max rows, max cols)
                const int pw = std::max(in.prev_w, in.w), ph = std::max(in.prev_h, in.h);
                const PyrDesc d = make_pyr_desc(pw, ph, t->cfg.lk_max_level > 1 ? t->cfg.lk_max_level : 1);
                PyrJob& a = C.pyr.h[2 * n_track];
                PyrJob& b = C.pyr.h[2 * n_track + 1];
                a.src = I.roi_gray + (set * 2 + (1 - in.cur_buf)) * P; a.sw = in.prev_w; a.sh = in.prev_h; a.spitch = in.prev_w;
                a.dst = I.pyr_prev + set * I.full.bytes; a.desc = d;
                b.src = c.dst; b.sw = in.w; b.sh = in.h; b.spitch = in.w;
                b.dst = I.pyr_cur + set * I.full.bytes; b.desc = d;
                LkGroup& G = C.lk_t.h[n_track];
                memset(&G, 0, sizeof(G));
                G.pyrA = a.dst; G.pyrB = b.dst; G.desc = d;
                G.ptsA = I.pts.pts + set * cap; G.ptsB = I.pts.lk_out + set * cap; G.status = I.pts.status + set * cap;
                G.n = I.pts.n + set;
                C.act_track.h[set] = 1;
                max_pw = std::max(max_pw, pw); max_ph = std::max(max_ph, ph); max_lv = std::max(max_lv, d.n_levels);
                n_track++;
            }
            // detection job (:418-446)
            ErodeJob& e = C.erode.h[j];
            e.tmp = I.roi_mask_tmp + set * P; e.dst = I.roi_mask_er + set * P;
            e.w = in.w; e.h = in.h; e.k = 5;
            if (in.label_bit >= 0) {       // full_mask(rect) read in place from the label image of this step
                e.src = t->lab_ptr[par] + (size_t)stream * t->lab_stride[par] + (size_t)in.y * t->lab_pitch[par] + in.x;
                e.spitch = t->lab_pitch[par]; e.label_bit = in.label_bit;
            } else {
                e.src = in.mask_off >= 0 ? C.d_mask_stage + in.mask_off : I.roi_mask + set * P;
                e.spitch = in.w; e.label_bit = -1;
            }
            GfttJob& J = C.gftt.h[j];
            memset(&J, 0, sizeof(J));
            J.img = c.dst; J.img_pitch = in.w; J.w = in.w; J.h = in.h;
            J.region_mask = e.dst; J.region_pitch = in.w;
            gftt_job_bind_scratch(&J, I.gsc, (int)set);
            J.pts = I.pts.pts + set * cap; J.ids = I.pts.ids + set * cap; J.track_cnt = I.pts.track_cnt + set * cap;
            J.n = I.pts.n + set; J.next_id = t->d_next_id + stream;
            J.max_cnt = t->cfg.max_dynamic_cnt; J.min_needed = 1;
            J.disc_radius = t->cfg.min_dynamic_dist; J.min_dist = (float)t->cfg.min_dynamic_dist; J.quality = 0.01;
            J.err = t->d_err + par;
            // stereo job: TrackRightByPad — full images, points offset by rect.tl()
            if (!stereo) continue;
            LkGroup& R = C.lk_s.h[n_stereo++];
            memset(&R, 0, sizeof(R));
            R.pyrA = left_pyr; R.pyrB = right_pyr; R.desc = t->desc;
            R.ptsA = I.pts.pts + set * cap; R.ptsB = I.pts.rpts + set * cap; R.status = I.pts.rstatus + set * cap;
            R.n = I.pts.n + set; R.offx = (float)in.x; R.offy = (float)in.y;
        }
    }

    // host -> device on the upload stream (all H2D traffic stays in one FIFO; the compute stream never queues a copy
    // behind the next frame's images): the packed masks and every descriptor array of this call in one copy each
    if (mask_used > 0) DVFE_CUDA(cudaMemcpyAsync(C.d_mask_stage, C.h_mask_stage, mask_used, cudaMemcpyHostToDevice, t->cs));
    if (nv > 0 || any_clear) DVFE_CHECK(C.arena.push(t->cs));
    if (mask_used > 0 || nv > 0 || any_clear) {
        DVFE_CUDA(cudaEventRecord(C.ev_up, t->cs));
        DVFE_CUDA(cudaStreamWaitEvent(st, C.ev_up, 0));
    }
    const size_t set0 = (size_t)s0 * MI;
    const int n_sets = (s1 - s0) * MI;
    if (nv > 0) {
        // views of the point sets of streams [s0, s1)
        PointSetArrays V = I.pts;
        const size_t o = set0 * cap;
        V.pts += o; V.lk_out += o; V.un += o; V.vel += o; V.ids += o; V.track_cnt += o; V.status += o; V.rpts += o;
        V.rstatus += o; V.rprev_un += o; V.rprev_valid += o; V.n += set0;

        DVFE_CHECK(launch_crop_jobs(C.crop.d, nv, max_rw, max_rh, st));
        // inst.TrackLeft(roi_gray_padded, prev_roi_gray_padded): previous-box crop -> current-box crop (:381-413)
        DVFE_CHECK(launch_build_pyramids_jobs(C.pyr.d, 2 * n_track, max_pw, max_ph, max_lv, st));
        DVFE_CHECK(launch_lk(C.lk_t.d, n_track, cap, t->cfg.lk_max_level, t->cfg.flow_back, st));
        DVFE_CHECK(launch_compact(V, n_sets, cap, st, C.act_track.d + set0));
        // ErodeMask(roi mask, 5) + discs(min_dynamic_dist) + goodFeaturesToTrack on the ROI + ids (:418-446)
        DVFE_CHECK(launch_erode_jobs(C.erode.d, nv, max_rw, max_rh, st));
        DVFE_CHECK(launch_gftt(C.gftt.d, nullptr, nv, max_rw, max_rh, cap, st));
        // UndistortedPointsWithAddOffset(cam0) + PtsVelocity(curr_time - last_time) (:448-457), each stream with the cameras of
        // its background step: the camera table is only rewritten ahead of the next step's kernels
        DVFE_CHECK(launch_left_post(V, n_sets, cap, t->d_cam + s0, MI, C.dt.d + set0, C.offs.d + set0, st, C.act_vis.d + set0));
        // TrackRightByPad + RightUndistortedPts + RightPtsVelocity (:462-471), then the Output() records
        if (n_stereo > 0) DVFE_CHECK(launch_lk(C.lk_s.d, n_stereo, cap, t->cfg.lk_max_level, t->cfg.flow_back, st));
        DVFE_CHECK(launch_inst_post_pack(V, n_sets, cap, t->d_cam + B + s0, MI, C.dt.d + set0, C.act_vis.d + set0, stereo_now ? 1 : 0,
                                         partial ? C.lane.d + set0 : nullptr, C.inst_id.d + set0, C.d_out + o, C.d_n + set0, st));
        C.has_records = true;
    }
    if (any_clear) DVFE_CHECK(launch_clear_sets(I.pts.n + set0, C.clear_flags.d + set0, n_sets, st));
    if (nv > 0) {
        // records home: on the download stream when deferred (the next step's kernels do not queue behind the copy)
        cudaStream_t os = defer ? t->ds : st;
        if (defer) {
            DVFE_CUDA(cudaEventRecord(C.ev_packed, st));
            DVFE_CUDA(cudaStreamWaitEvent(os, C.ev_packed, 0));
        }
        const size_t o = set0 * cap;
        DVFE_CUDA(cudaMemcpyAsync(C.h_n + set0, C.d_n + set0, n_sets * sizeof(int), cudaMemcpyDeviceToHost, os));
        DVFE_CUDA(cudaMemcpyAsync(C.h_n + NS, t->d_err + par, sizeof(int), cudaMemcpyDeviceToHost, os));
        DVFE_CUDA(cudaMemcpyAsync(C.h_out + o, C.d_out + o, (size_t)n_sets * cap * sizeof(dvfe_inst_obs),
                                  cudaMemcpyDeviceToHost, os));
    }

    // host bookkeeping after the frame: ManageInstances (:474), PostProcess (:479-481), the Output() plan (:521-577)
    for (int stream = s0; stream < s1; stream++) {
        if (!exist[stream - s0]) continue;
        InstStream& S = I.streams[stream];
        const size_t base_set = (size_t)stream * MI;
        manage_instances(S);
        for (auto& kv : S.insts) {
            InstHost& in = kv.second;
            if (in.lost_num > 0) continue;
            in.prev_w = in.roi_w; in.prev_h = in.roi_h;          // prev_roi_gray = roi_gray
        }
        // Output(): lost_num == 0 && is_curr_visible, ascending instance id, ascending feature id
        for (auto& kv : S.insts) {
            const InstHost& in = kv.second;
            if (in.lost_num > 0 || !in.visible) continue;
            C.plan.push_back({stream, (int)(base_set + in.slot), in.disp, in.disp_pitch});
        }
        S.last_time = time_of[stream - s0];
    }
    if (defer) {
        DVFE_CUDA(cudaEventRecord(t->ev_inst[par], nv > 0 ? t->ds : st));
        t->inst_pending[par] = true;
        return DVFE_OK;
    }
    if (nv > 0 || any_clear || mask_used > 0) DVFE_CUDA(cudaStreamSynchronize(st));
    return t->finish_instances(par);
}

// Output() of a finished call: copy the records of the planned instances out of the pinned buffer
int dvfe_tracker::finish_instances(int par) {
    InstanceState& I = *inst;
    InstCall& C = I.call[par];
    for (int s = C.s0; s < C.s1; s++) I.streams[s].out.clear();
    for (const auto& e : C.plan) {
        std::vector<dvfe_inst_obs>& out = I.streams[e.stream].out;
        const size_t set = (size_t)e.set;
        const int n = C.has_records ? C.h_n[set] : 0;
        const size_t first = out.size();
        out.insert(out.end(), C.h_out + set * I.cap, C.h_out + set * I.cap + n);
        if (e.disp != nullptr)
            // feat->disp = prev_img.disp.at<float>(inst.curr_points[i]) (front_end/dynamic_tracker.cpp:547): a lookup in the
            // caller's full-size map with the ROI-LOCAL position, rounded to the nearest pixel (ties to even) as Mat::at(Point2f)
            // does.  A table lookup in a host input, done where the records land.
            for (size_t i = first; i < out.size(); i++) {
                const long col = lrint(out[i].uv[0]), row = lrint(out[i].uv[1]);
                out[i].disp = (double)*reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(e.disp) +
                                                                      (size_t)row * e.disp_pitch + (size_t)col * sizeof(float));
            }
    }
    if (C.has_records && C.h_n[(size_t)B * I.MI] != 0) {
        dvfe_set_error("corner detection on an instance ROI: more local maxima than the candidate buffer holds; the selection "
                       "of this frame was truncated");
        return DVFE_ERR_CAPACITY;
    }
    return DVFE_OK;
}

int grp_track_dynamic_async(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, const uint8_t* inv, size_t stride,
                            int pitch, const int* exist, const dvfe_inst_in* boxes, const int* n_boxes, const double* time0,
                            const uint8_t* stream_flags, unsigned flags);
int grp_insts_track(dvfe_tracker* t, int stream, const dvfe_inst_in* boxes, int n, double time0);
int grp_insts_track_batch(dvfe_tracker* t, const dvfe_inst_in* boxes, const int* n_boxes, const double* time0);
int grp_route(dvfe_tracker* t, int stream, dvfe_tracker** leaf, int* local);

static int insts_check(dvfe_tracker* t) {
    if (!t || !t->inst) {
        dvfe_set_error("insts_track: bad argument (max_instances must be > 0 at create)");
        return DVFE_ERR_INVALID;
    }
    if (t->frames == 0) {
        dvfe_set_error("insts_track: no frame has been uploaded yet (call dvfe_track_semantic_image first)");
        return DVFE_ERR_INVALID;
    }
    return DVFE_OK;
}

extern "C" int dvfe_insts_track(dvfe_tracker* t, int stream, const dvfe_inst_in* boxes, int n_boxes, double time0) {
    if (t && !t->groups.empty()) return grp_insts_track(t, stream, boxes, n_boxes, time0);
    DVFE_CHECK(insts_check(t));
    if (stream < 0 || stream >= t->B || n_boxes < 0 || (n_boxes > 0 && !boxes)) {
        dvfe_set_error("insts_track: bad argument");
        return DVFE_ERR_INVALID;
    }
    return insts_track_streams(t, stream, stream + 1, &boxes, &n_boxes, &time0, false);
}

extern "C" int dvfe_insts_track_batch(dvfe_tracker* t, const dvfe_inst_in* boxes, const int* n_boxes, const double* time0) {
    if (t && !t->groups.empty()) {
        if (!n_boxes || !time0) { dvfe_set_error("insts_track_batch: null argument"); return DVFE_ERR_INVALID; }
        return grp_insts_track_batch(t, boxes, n_boxes, time0);
    }
    DVFE_CHECK(insts_check(t));
    if (!n_boxes || !time0) { dvfe_set_error("insts_track_batch: null argument"); return DVFE_ERR_INVALID; }
    std::vector<const dvfe_inst_in*> of(t->B);
    size_t off = 0;
    for (int s = 0; s < t->B; s++) {
        if (n_boxes[s] < 0 || (n_boxes[s] > 0 && !boxes)) { dvfe_set_error("insts_track_batch: bad box count"); return DVFE_ERR_INVALID; }
        of[s] = boxes + off;
        off += (size_t)n_boxes[s];
    }
    return insts_track_streams(t, 0, t->B, of.data(), n_boxes, time0, false);
}

// One frame of dynamic mode for all streams, pipelined: TrackSemanticImage + InstsTrack are enqueued behind the previous
// step (two steps in flight); dvfe_wait() completes the oldest one, after which dvfe_get_features / dvfe_insts_output
// return its results.
extern "C" int dvfe_track_dynamic_async(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, const uint8_t* inv_merge_mask,
                                        size_t stream_stride, int pitch, const int* exist_inst, const dvfe_inst_in* boxes,
                                        const int* n_boxes, const double* time0) {
    return dvfe_track_dynamic_ex2(t, left, right, inv_merge_mask, stream_stride, pitch, exist_inst, boxes, n_boxes, time0, nullptr, 0u);
}

extern "C" int dvfe_track_dynamic_ex(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, const uint8_t* mask,
                                     size_t stream_stride, int pitch, const int* exist_inst, const dvfe_inst_in* boxes,
                                     const int* n_boxes, const double* time0, unsigned flags) {
    return dvfe_track_dynamic_ex2(t, left, right, mask, stream_stride, pitch, exist_inst, boxes, n_boxes, time0, nullptr, flags);
}

extern "C" int dvfe_track_dynamic_ex2(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, const uint8_t* mask,
                                      size_t stream_stride, int pitch, const int* exist_inst, const dvfe_inst_in* boxes,
                                      const int* n_boxes, const double* time0, const uint8_t* stream_flags, unsigned flags) {
    const bool labels = (flags & DVFE_DYN_LABELS) != 0;
    if (!t || !left || !time0 || !n_boxes || (!exist_inst && !labels)) { dvfe_set_error("track_dynamic: null argument"); return DVFE_ERR_INVALID; }
    const uint8_t* sf = nullptr;
    DVFE_CHECK(check_stream_flags(stream_flags, t->B, "track_dynamic", &sf));
    std::vector<const dvfe_inst_in*> of(t->B);
    size_t off = 0;
    for (int s = 0; s < t->B; s++) {
        if (n_boxes[s] < 0 || (n_boxes[s] > 0 && !boxes)) { dvfe_set_error("track_dynamic_async: bad box count"); return DVFE_ERR_INVALID; }
        of[s] = boxes + off;
        off += (size_t)n_boxes[s];
    }
    if (!t->groups.empty()) {
        // every group's boxes are checked before the first group enqueues anything
        for (size_t g = 0; g < t->groups.size(); g++) {
            dvfe_tracker* leaf = t->groups[g];
            const int f = t->group_first[g];
            if (leaf->inst) DVFE_CHECK(insts_validate(leaf, 0, leaf->B, of.data() + f, n_boxes + f, labels, sf ? sf + f : nullptr));
        }
        return grp_track_dynamic_async(t, left, right, mask, stream_stride, pitch, exist_inst, boxes, n_boxes, time0, sf, flags);
    }
    if (!t->inst) { dvfe_set_error("track_dynamic_async: max_instances must be > 0 at create"); return DVFE_ERR_INVALID; }
    if (pitch < t->W * t->in_ch) { dvfe_set_error("track_dynamic_async: bad pitch"); return DVFE_ERR_INVALID; }
    DVFE_CHECK(insts_validate(t, 0, t->B, of.data(), n_boxes, labels, sf));
    return leaf_track_dynamic(t, t->slab(left, right, mask, stream_stride, pitch), exist_inst, of.data(), n_boxes, time0, sf, flags);
}

int leaf_validate_boxes(dvfe_tracker* t, const dvfe_inst_in* const* boxes_of, const int* n_boxes, bool labels, const uint8_t* sflags) {
    if (!t->inst) { dvfe_set_error("track_dynamic: max_instances must be > 0 at create"); return DVFE_ERR_INVALID; }
    return insts_validate(t, 0, t->B, boxes_of, n_boxes, labels, sflags);
}

int leaf_track_dynamic(dvfe_tracker* t, const StepSources& src, const int* exist_inst, const dvfe_inst_in* const* boxes_of,
                       const int* n_boxes, const double* time0, const uint8_t* sf, unsigned flags) {
    const bool labels = (flags & DVFE_DYN_LABELS) != 0;
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    // SetMaskAndRoi: exist_inst = !boxes2d.empty(); a skipped stream's exist_inst is not read
    std::vector<int> exist(t->B);
    for (int s = 0; s < t->B; s++)
        exist[s] = (sf && (sf[s] & DVFE_FRAME_SKIP)) ? 0 : labels ? (n_boxes[s] > 0 ? 1 : 0) : exist_inst[s];
    DVFE_CHECK(t->semantic_submit(src, exist.data(), time0, flags, sf));
    return insts_track_streams(t, 0, t->B, boxes_of, n_boxes, time0, true, labels);
}

extern "C" int dvfe_insts_output(dvfe_tracker* t, int stream, dvfe_inst_obs* out, int cap, int* n_out) {
    if (t && !t->groups.empty()) {
        dvfe_tracker* leaf; int local;
        DVFE_CHECK(grp_route(t, stream, &leaf, &local));
        return dvfe_insts_output(leaf, local, out, cap, n_out);
    }
    if (!t || !t->inst || stream < 0 || stream >= t->B || !n_out) {
        dvfe_set_error("insts_output: bad argument");
        return DVFE_ERR_INVALID;
    }
    const std::vector<dvfe_inst_obs>& v = t->inst->streams[stream].out;
    *n_out = (int)v.size();
    if ((int)v.size() > cap) { dvfe_set_error("insts_output: %d records, capacity %d", (int)v.size(), cap); return DVFE_ERR_CAPACITY; }
    if (!v.empty() && out) memcpy(out, v.data(), v.size() * sizeof(dvfe_inst_obs));
    return DVFE_OK;
}

extern "C" int dvfe_insts_table(dvfe_tracker* t, int stream, dvfe_inst_info* out, int cap, int* n_out) {
    if (t && !t->groups.empty()) {
        dvfe_tracker* leaf; int local;
        DVFE_CHECK(grp_route(t, stream, &leaf, &local));
        return dvfe_insts_table(leaf, local, out, cap, n_out);
    }
    if (!t || !t->inst || stream < 0 || stream >= t->B || !n_out) {
        dvfe_set_error("insts_table: bad argument");
        return DVFE_ERR_INVALID;
    }
    const InstStream& S = t->inst->streams[stream];
    *n_out = (int)S.insts.size();
    if (*n_out > cap) { dvfe_set_error("insts_table: %d instances, capacity %d", *n_out, cap); return DVFE_ERR_CAPACITY; }
    int i = 0;
    for (const auto& kv : S.insts) {
        const InstHost& in = kv.second;
        if (out) out[i] = dvfe_inst_info{in.track_id, in.lost_num, in.visible ? 1 : 0, in.has_box ? 1 : 0, in.x, in.y, in.w, in.h};
        i++;
    }
    return DVFE_OK;
}
