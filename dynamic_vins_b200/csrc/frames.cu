// Per-camera frame descriptors (dvfe_track_frames / _semantic_frames / _dynamic_frames, include/dvfe.h): the steps of the slab
// entry points, with a source table built camera by camera instead of base + s * stride.  The whole call is validated before
// any stream group enqueues, so a rejected call changes nothing.
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

enum FrameMode { FM_RAW, FM_SEMANTIC, FM_DYNAMIC };

// The slab call a descriptor array stands for: its stream flags, times and exist_inst
struct FrameStep {
    std::vector<uint8_t> sflags;
    std::vector<double> time0;
    std::vector<int> exist;
    bool any_right = false;          // some present frame has a right image (and the tracker is stereo): a stereo step
};

int check_frames(dvfe_tracker* t, const dvfe_frame* frames, unsigned flags, FrameMode mode, const int* n_boxes, const char* who,
                 FrameStep* fs) {
    if (!t || !frames) { dvfe_set_error("%s: null tracker or frames", who); return DVFE_ERR_INVALID; }
    const unsigned known = mode == FM_RAW ? DVFE_STEP_DEVICE_INPUT
                         : mode == FM_SEMANTIC ? DVFE_DYN_DEVICE_INPUT : (DVFE_DYN_DEVICE_INPUT | DVFE_DYN_LABELS);
    if (flags & ~known) { dvfe_set_error("%s: unknown flags 0x%x", who, flags); return DVFE_ERR_INVALID; }
    if (mode == FM_DYNAMIC && !n_boxes) { dvfe_set_error("%s: n_boxes is null", who); return DVFE_ERR_INVALID; }
    const dvfe_tracker* leaf0 = t->groups.empty() ? t : t->groups[0];
    const int B = t->B, row = t->W * leaf0->in_ch;
    const bool labels = (flags & DVFE_DYN_LABELS) != 0;
    fs->sflags.assign(B, 0);
    fs->time0.assign(B, 0.0);
    fs->exist.assign(B, 0);
    fs->any_right = false;
    for (int s = 0; s < B; s++) {
        const dvfe_frame& f = frames[s];
        if (f.flags & ~DVFE_FRAME_RESET) { dvfe_set_error("%s: stream %d: invalid frame flags 0x%x", who, s, f.flags); return DVFE_ERR_INVALID; }
        if (!f.left) {
            if (f.flags & DVFE_FRAME_RESET) { dvfe_set_error("%s: stream %d: DVFE_FRAME_RESET without a frame", who, s); return DVFE_ERR_INVALID; }
            continue;
        }
        if (f.pitch < row) { dvfe_set_error("%s: stream %d: pitch %d < %d", who, s, f.pitch, row); return DVFE_ERR_INVALID; }
        if (mode != FM_RAW) {
            if (f.mask && f.mask_pitch < t->W) {
                dvfe_set_error("%s: stream %d: mask_pitch %d < %d", who, s, f.mask_pitch, t->W);
                return DVFE_ERR_INVALID;
            }
            const bool needs_mask = labels ? n_boxes[s] > 0 : f.exist_inst != 0;
            if (needs_mask && !f.mask) {
                dvfe_set_error("%s: stream %d: %s but no mask", who, s, labels ? "boxes" : "exist_inst set");
                return DVFE_ERR_INVALID;
            }
        }
        fs->any_right = fs->any_right || (t->cfg.stereo && f.right);
    }
    for (int s = 0; s < B; s++) {
        const dvfe_frame& f = frames[s];
        if (!f.left) { fs->sflags[s] = DVFE_FRAME_SKIP; continue; }
        fs->sflags[s] = (uint8_t)(f.flags | (fs->any_right && !f.right ? DVFE_FRAME_NO_RIGHT : 0u));
        fs->time0[s] = f.time0;
        fs->exist[s] = f.exist_inst;
    }
    return DVFE_OK;
}

// image c of every stream is present, at one pitch and one stride: the table is that of a slab
void find_slab(StepSources* src, int c, int H) {
    const std::vector<ImgSrc>& v = src->img[c];
    const size_t n = v.size();
    for (const ImgSrc& e : v)
        if (!e.ptr || e.pitch != v[0].pitch) return;
    const ptrdiff_t d = n > 1 ? v[1].ptr - v[0].ptr : (ptrdiff_t)v[0].pitch * H;
    if (d <= 0) return;
    for (size_t s = 1; s < n; s++)
        if (v[s].ptr != v[0].ptr + (ptrdiff_t)s * d) return;
    src->uniform[c] = true;
    src->stride[c] = (size_t)d;
}

StepSources frame_sources(const dvfe_frame* f, int n, const FrameStep& fs, bool masks, int H) {
    StepSources src;
    for (int c = 0; c < 3; c++) src.img[c].assign(n, ImgSrc{nullptr, 0});
    for (int s = 0; s < n; s++) {
        if (!f[s].left) continue;
        src.img[0][s] = ImgSrc{f[s].left, f[s].pitch};
        if (fs.any_right && f[s].right) src.img[1][s] = ImgSrc{f[s].right, f[s].pitch};
        if (masks && f[s].mask) src.img[2][s] = ImgSrc{f[s].mask, f[s].mask_pitch};
    }
    for (int c = 0; c < 3; c++) find_slab(&src, c, H);
    return src;
}

int track_frames(dvfe_tracker* t, const dvfe_frame* frames, const dvfe_inst_in* boxes, const int* n_boxes, unsigned flags,
                 FrameMode mode, const char* who) {
    FrameStep fs;
    DVFE_CHECK(check_frames(t, frames, flags, mode, n_boxes, who, &fs));
    const bool device = (flags & DVFE_STEP_DEVICE_INPUT) != 0;
    std::vector<dvfe_tracker*> leaves = t->groups;
    std::vector<int> first = t->group_first;
    if (leaves.empty()) { leaves.assign(1, t); first = {0, t->B}; }
    std::vector<const dvfe_inst_in*> of;
    if (mode == FM_DYNAMIC) {
        of.resize(t->B);
        size_t off = 0;
        for (int s = 0; s < t->B; s++) {
            if (n_boxes[s] < 0 || (n_boxes[s] > 0 && !boxes)) { dvfe_set_error("%s: stream %d: bad box count", who, s); return DVFE_ERR_INVALID; }
            of[s] = boxes + off;
            off += (size_t)n_boxes[s];
        }
        for (size_t g = 0; g < leaves.size(); g++) {
            const int f = first[g];
            DVFE_CHECK(leaf_validate_boxes(leaves[g], of.data() + f, n_boxes + f, (flags & DVFE_DYN_LABELS) != 0, fs.sflags.data() + f));
        }
    }
    // every group submits a step, also one whose streams are all skipped, so that each dvfe_wait still pairs with one step per group
    for (size_t g = 0; g < leaves.size(); g++) {
        dvfe_tracker* leaf = leaves[g];
        const int f = first[g];
        const uint8_t* sf = nullptr;                      // null when the group's flags are all 0: the plain step
        DVFE_CHECK(check_stream_flags(fs.sflags.data() + f, leaf->B, who, &sf));
        const StepSources src = frame_sources(frames + f, leaf->B, fs, mode != FM_RAW, leaf->H);
        if (mode == FM_RAW) {
            DVFE_CHECK(leaf_track(leaf, src, fs.time0.data() + f, sf, device));
        } else if (mode == FM_SEMANTIC) {
            DVFE_CUDA(cudaSetDevice(leaf->cfg.device));
            DVFE_CHECK(leaf->semantic_submit(src, fs.exist.data() + f, fs.time0.data() + f, flags, sf));
        } else {
            DVFE_CHECK(leaf_track_dynamic(leaf, src, fs.exist.data() + f, of.data() + f, n_boxes + f, fs.time0.data() + f, sf, flags));
        }
    }
    return DVFE_OK;
}

}  // namespace

extern "C" int dvfe_track_frames(dvfe_tracker* t, const dvfe_frame* frames, unsigned flags) {
    return track_frames(t, frames, nullptr, nullptr, flags, FM_RAW, "dvfe_track_frames");
}

extern "C" int dvfe_track_semantic_frames(dvfe_tracker* t, const dvfe_frame* frames, unsigned flags) {
    return track_frames(t, frames, nullptr, nullptr, flags, FM_SEMANTIC, "dvfe_track_semantic_frames");
}

extern "C" int dvfe_track_dynamic_frames(dvfe_tracker* t, const dvfe_frame* frames, const dvfe_inst_in* boxes, const int* n_boxes,
                                         unsigned flags) {
    return track_frames(t, frames, boxes, n_boxes, flags, FM_DYNAMIC, "dvfe_track_dynamic_frames");
}
