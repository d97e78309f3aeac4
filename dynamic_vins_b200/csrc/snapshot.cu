// Stream snapshots (dvfe_export_stream / dvfe_import_stream): everything the next step of one stream reads from earlier frames, as
// one self-describing host blob, and back into any slot of a tracker with the same front-end parameters (DESIGN.md §2):
//
//   SnapHeader | SnapInst x n_inst | payload (16-byte aligned) | CRC-32 (zlib's) of all bytes before it
//
// The payload is the device state, in a section order both sides derive from the header alone: the background point set (count,
// id counter, ids, track_cnt, last points, prev_un, right_prev_un, right_prev_valid; whole arrays of max_cnt entries), the interior
// of level 0 of the stream's previous left pyramid (W x H, when the stream has had a frame), then per instance in ascending track id
// its point set (the same arrays, max_dynamic_cnt entries) and its previous ROI crop (prev_w x prev_h).  One gather kernel copies
// those pieces into a staging buffer, one copy brings it home; an import copies it back and scatters it with the same kernel, then
// rebuilds the previous left pyramid from level 0 with the frame step's own pyramid kernels.
#include <string.h>

#include <vector>

#include "kernels.cuh"
#include "state.cuh"
#include "tracker.h"

#define DVFE_CHECK(call)                 \
    do {                                 \
        int rc__ = (call);               \
        if (rc__ != DVFE_OK) return rc__; \
    } while (0)

int grp_route(dvfe_tracker* t, int stream, dvfe_tracker** leaf, int* local);

namespace {
const uint32_t kSnapMagic = 0x53535644u;            // "DVSS"
const uint32_t kSnapVersion = 1;
const int kCompat = 11;                              // front-end fields that must match (compat_fields)

struct SnapHeader {
    uint32_t magic, version;
    uint64_t total_bytes;                            // the whole blob, CRC included
    int32_t compat[kCompat];
    int32_t has_image;                               // the payload holds the stream's last left image
    int32_t n_inst;                                  // SnapInst records after the header
    int32_t reserved;
    double prev_time;                                // FeatureTracker prev_time
    double last_time;                                // InstsFeatManager last_time (0 without instances)
    CamParams cam[2];                                // the stream's cam0 / cam1 as the post kernels read them
    uint64_t payload_bytes;
};

void compat_fields(const dvfe_config& c, int32_t* f) {
    const int32_t v[kCompat] = {c.width, c.height, c.stereo, c.max_cnt, c.min_dist, c.max_dynamic_cnt, c.min_dynamic_dist,
                                c.flow_back, c.use_mask_morphology, c.mask_morphology_size, c.lk_max_level};
    memcpy(f, v, sizeof(v));
}
const char* const kCompatNames[kCompat] = {"width", "height", "stereo", "max_cnt", "min_dist", "max_dynamic_cnt", "min_dynamic_dist",
                                           "flow_back", "use_mask_morphology", "mask_morphology_size", "lk_max_level"};

size_t payload_offset(int n_inst) { return (sizeof(SnapHeader) + (size_t)n_inst * sizeof(SnapInst) + 15) & ~(size_t)15; }

uint32_t crc32(const uint8_t* p, size_t n) {
    static uint32_t table[256];
    static const bool init = [] {
        for (uint32_t i = 0; i < 256; i++) {
            uint32_t c = i;
            for (int k = 0; k < 8; k++) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
            table[i] = c;
        }
        return true;
    }();
    (void)init;
    uint32_t c = 0xFFFFFFFFu;
    for (size_t i = 0; i < n; i++) c = table[(c ^ p[i]) & 0xFF] ^ (c >> 8);
    return c ^ 0xFFFFFFFFu;
}

// one piece of device state: `rows` rows of `row` bytes at `pitch` on the device, dense at `off` in the staging buffer
struct SnapSeg {
    uint8_t* dev;
    uint32_t off, pitch, row, rows;
};
#define SNAP_SEGS 160                                // per launch: the table is a kernel parameter (< 4 KB)
struct SnapSegs {
    SnapSeg s[SNAP_SEGS];
};

// to_stage = 1: device state -> staging (export), 0: staging -> device state (import).  One segment per grid row; 16-byte vectors
// where the segment allows them.
__global__ void __launch_bounds__(256) k_snap_copy(SnapSegs t, uint8_t* __restrict__ stage, int to_stage) {
    const SnapSeg g = t.s[blockIdx.y];
    uint8_t* sp = stage + g.off;
    const size_t step = (size_t)gridDim.x * blockDim.x;
    if ((((size_t)g.dev | g.off | g.pitch | g.row) & 15) == 0) {
        const uint32_t vrow = g.row / 16;
        const size_t nv = (size_t)vrow * g.rows;
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += step) {
            uint4* d = reinterpret_cast<uint4*>(g.dev + (i / vrow) * g.pitch) + i % vrow;
            uint4* s = reinterpret_cast<uint4*>(sp) + i;
            if (to_stage) *s = *d;
            else *d = *s;
        }
    } else {
        const size_t nb = (size_t)g.row * g.rows;
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nb; i += step) {
            uint8_t* d = g.dev + (i / g.row) * g.pitch + i % g.row;
            if (to_stage) sp[i] = *d;
            else *d = sp[i];
        }
    }
}

struct SnapLayout {
    std::vector<SnapSeg> segs;
    std::vector<int> counts;                         // the segments that hold a point count (checked on import)
    size_t bytes = 0;
    void add(void* dev, size_t pitch, size_t row, size_t rows) {
        bytes = (bytes + 15) & ~(size_t)15;
        segs.push_back(SnapSeg{(uint8_t*)dev, (uint32_t)bytes, (uint32_t)pitch, (uint32_t)row, (uint32_t)rows});
        bytes += row * rows;
    }
    void add_array(void* dev, size_t n) { add(dev, n, n, 1); }
    // what a point set carries into the next frame (the other arrays are rewritten by every frame before they are read)
    // S null: sizes only.  id_counter: the background's, shared with the stream's instances
    void add_set(const PointSetArrays* S, size_t set, int cap, bool with_counter, uint32_t* id_counter) {
        const size_t o = set * cap;
        const bool d = S != nullptr;
        counts.push_back((int)segs.size());
        add_array(d ? S->n + set : nullptr, sizeof(int));
        if (with_counter) add_array(d ? id_counter : nullptr, sizeof(uint32_t));
        add_array(d ? S->ids + o : nullptr, cap * sizeof(uint32_t));
        add_array(d ? S->track_cnt + o : nullptr, cap * sizeof(int32_t));
        add_array(d ? S->pts + o : nullptr, cap * sizeof(float2));
        add_array(d ? S->un + o : nullptr, cap * sizeof(float2));
        add_array(d ? S->rprev_un + o : nullptr, cap * sizeof(float2));
        add_array(d ? S->rprev_valid + o : nullptr, (size_t)cap);
    }
};

// dev: where each instance's state lives; null: sizes only (the device pointers stay null)
SnapLayout snap_layout(const dvfe_tracker* t, int stream, bool has_image, const std::vector<SnapInst>& recs,
                       const std::vector<SnapInstDev>* dev) {
    SnapLayout L;
    const bool d = dev != nullptr;
    L.add_set(d ? &t->bg : nullptr, (size_t)stream, t->cap, true, t->d_next_id + stream);
    if (has_image) {
        const PyrLevel& L0 = t->desc.lv[0];
        uint8_t* px = t->left_slot(t->frames + 2) + (size_t)stream * t->desc.bytes + L0.offset + (size_t)DVFE_PADY * L0.pitch + DVFE_PADX;
        L.add(d ? px : nullptr, (size_t)L0.pitch, (size_t)t->W, (size_t)t->H);
    }
    for (size_t i = 0; i < recs.size(); i++) {
        L.add_set(d ? &t->inst_points() : nullptr, d ? (*dev)[i].set : 0, t->cfg.max_dynamic_cnt, false, nullptr);
        if (recs[i].prev_w > 0 && recs[i].prev_h > 0)
            L.add_array(d ? (*dev)[i].crop : nullptr, (size_t)recs[i].prev_w * recs[i].prev_h);
    }
    return L;
}

// the staging buffer at its largest: an image and every instance slot with a full-size crop
int snap_stage(dvfe_tracker* t) {
    if (t->d_snap) return DVFE_OK;
    std::vector<SnapInst> recs((size_t)(t->inst ? t->cfg.max_instances : 0));
    for (SnapInst& r : recs) { memset(&r, 0, sizeof(r)); r.prev_w = t->W; r.prev_h = t->H; }
    const size_t bytes = snap_layout(t, 0, true, recs, nullptr).bytes;
    DVFE_CUDA(cudaMalloc((void**)&t->d_snap, bytes));
    DVFE_CUDA(cudaMemset(t->d_snap, 0, bytes));      // the alignment gaps between segments: a blob is a function of the state
    return DVFE_OK;
}

int snap_copy(const SnapLayout& L, uint8_t* stage, int to_stage, cudaStream_t st) {
    for (size_t first = 0; first < L.segs.size(); first += SNAP_SEGS) {
        const size_t n = L.segs.size() - first < SNAP_SEGS ? L.segs.size() - first : SNAP_SEGS;
        SnapSegs tab;
        memset(&tab, 0, sizeof(tab));
        size_t most = 0;
        for (size_t i = 0; i < n; i++) {
            tab.s[i] = L.segs[first + i];
            const size_t b = (size_t)tab.s[i].row * tab.s[i].rows;
            most = b > most ? b : most;
        }
        size_t blocks = (most / 16 + 255) / 256;
        blocks = blocks < 1 ? 1 : blocks > 512 ? 512 : blocks;
        DVFE_LAUNCH(k_snap_copy, dim3((unsigned)blocks, (unsigned)n), dim3(256), 0, st, tab, stage, to_stage);
    }
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

int in_flight(const dvfe_tracker* t, const char* who) {
    if (t->completed < t->frames) {
        dvfe_set_error("%s: %ld step(s) in flight; wait for them first", who, t->frames - t->completed);
        return DVFE_ERR_INVALID;
    }
    return DVFE_OK;
}

int leaf_export(dvfe_tracker* t, int stream, uint8_t* blob, size_t cap, size_t* n_bytes) {
    DVFE_CHECK(in_flight(t, "export_stream"));
    std::vector<SnapInst> recs;
    std::vector<SnapInstDev> dev;
    double last_time = 0.0;
    if (t->inst) t->insts_export(stream, &recs, &dev, &last_time);
    const bool has_image = t->had_frame[stream] != 0;
    const SnapLayout L = snap_layout(t, stream, has_image, recs, &dev);
    const size_t poff = payload_offset((int)recs.size()), total = poff + L.bytes + 4;
    *n_bytes = total;
    if (!blob) return DVFE_OK;
    if (cap < total) { dvfe_set_error("export_stream: the snapshot takes %zu bytes, capacity %zu", total, cap); return DVFE_ERR_CAPACITY; }
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    DVFE_CHECK(snap_stage(t));
    DVFE_CHECK(snap_copy(L, t->d_snap, 1, t->st));
    DVFE_CUDA(cudaMemcpyAsync(blob + poff, t->d_snap, L.bytes, cudaMemcpyDeviceToHost, t->st));
    DVFE_CUDA(cudaStreamSynchronize(t->st));
    SnapHeader h;
    memset(&h, 0, sizeof(h));
    h.magic = kSnapMagic; h.version = kSnapVersion; h.total_bytes = total;
    compat_fields(t->cfg, h.compat);
    h.has_image = has_image ? 1 : 0;
    h.n_inst = (int32_t)recs.size();
    h.prev_time = t->prev_time[stream];
    h.last_time = last_time;
    h.cam[0] = t->cams[stream];
    h.cam[1] = t->cams[(size_t)t->B + stream];
    h.payload_bytes = L.bytes;
    memset(blob, 0, poff);
    memcpy(blob, &h, sizeof(h));
    if (!recs.empty()) memcpy(blob + sizeof(h), recs.data(), recs.size() * sizeof(SnapInst));
    const uint32_t crc = crc32(blob, total - 4);
    memcpy(blob + total - 4, &crc, 4);
    return DVFE_OK;
}

int bad_blob(const char* why) {
    dvfe_set_error("import_stream: %s", why);
    return DVFE_ERR_INVALID;
}

int leaf_import(dvfe_tracker* t, int stream, const uint8_t* blob, size_t n) {
    DVFE_CHECK(in_flight(t, "import_stream"));
    // ---- everything is checked before anything changes ----
    SnapHeader h;
    if (n < sizeof(h) + 4) return bad_blob("truncated snapshot");
    memcpy(&h, blob, sizeof(h));
    if (h.magic != kSnapMagic) return bad_blob("not a stream snapshot (bad magic number)");
    if (h.version != kSnapVersion) {
        dvfe_set_error("import_stream: snapshot format version %u, this library reads version %u", h.version, kSnapVersion);
        return DVFE_ERR_INVALID;
    }
    if (h.total_bytes != n) {
        dvfe_set_error("import_stream: the snapshot has %llu bytes, %zu given (truncated?)", (unsigned long long)h.total_bytes, n);
        return DVFE_ERR_INVALID;
    }
    uint32_t crc;
    memcpy(&crc, blob + n - 4, 4);
    if (crc32(blob, n - 4) != crc) return bad_blob("CRC-32 mismatch (corrupted snapshot)");
    int32_t want[kCompat];
    compat_fields(t->cfg, want);
    for (int i = 0; i < kCompat; i++)
        if (h.compat[i] != want[i]) {
            dvfe_set_error("import_stream: snapshot %s = %d, this tracker's is %d", kCompatNames[i], h.compat[i], want[i]);
            return DVFE_ERR_INVALID;
        }
    const int MI = t->inst ? t->cfg.max_instances : 0;
    if (h.n_inst < 0 || h.n_inst > MI) {
        dvfe_set_error("import_stream: the snapshot has %d instances, this tracker's max_instances is %d", h.n_inst, MI);
        return DVFE_ERR_INVALID;
    }
    if (h.has_image != 0 && h.has_image != 1) return bad_blob("bad header");
    const size_t poff = payload_offset(h.n_inst);
    if (poff + h.payload_bytes + 4 != n) return bad_blob("section sizes do not add up");
    std::vector<SnapInst> recs((size_t)h.n_inst);
    if (h.n_inst > 0) memcpy(recs.data(), blob + sizeof(h), recs.size() * sizeof(SnapInst));
    for (size_t i = 0; i < recs.size(); i++) {
        const SnapInst& r = recs[i];
        if ((i > 0 && r.track_id <= recs[i - 1].track_id) || r.prev_w < 0 || r.prev_w > t->W || r.prev_h < 0 || r.prev_h > t->H ||
            r.lost_num < 0)
            return bad_blob("bad instance record");
    }
    const SnapLayout sizes = snap_layout(t, stream, h.has_image != 0, recs, nullptr);
    if (sizes.bytes != h.payload_bytes) return bad_blob("section sizes do not add up");
    for (size_t i = 0; i < sizes.counts.size(); i++) {
        int c;
        memcpy(&c, blob + poff + sizes.segs[(size_t)sizes.counts[i]].off, sizeof(c));
        if (c < 0 || c > (i == 0 ? t->cap : t->cfg.max_dynamic_cnt)) return bad_blob("point count out of range");
    }
    // ---- apply ----
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    DVFE_CHECK(snap_stage(t));
    std::vector<SnapInstDev> dev;
    if (t->inst) t->insts_import(stream, recs, h.last_time, &dev);
    const SnapLayout L = snap_layout(t, stream, h.has_image != 0, recs, &dev);
    DVFE_CUDA(cudaMemcpyAsync(t->d_snap, blob + poff, L.bytes, cudaMemcpyHostToDevice, t->st));
    DVFE_CHECK(snap_copy(L, t->d_snap, 0, t->st));
    if (h.has_image) {
        // the previous left pyramid of the next step, from its level-0 interior: the border and the upper levels as the step built them
        PyrImgSet set;
        set.src[0] = nullptr; set.src[1] = nullptr;
        set.dst[0] = t->left_slot(t->frames + 2) + (size_t)stream * t->desc.bytes; set.dst[1] = nullptr;
        set.src_stride = 0; set.dst_stride = t->desc.bytes; set.per_set = 1;
        DVFE_CHECK(launch_build_pyramids(set, 1, t->desc, 0, t->st, DVFE_L0_INTERIOR));
    }
    DVFE_CUDA(cudaStreamSynchronize(t->st));
    t->prev_time[stream] = h.prev_time;
    t->had_frame[stream] = (uint8_t)h.has_image;
    if (h.has_image) t->prev_loaded = true;
    t->tc_valid[stream] = 0;                 // the cached templates belong to the points that were just replaced
    t->tcache_valid = false;
    t->cams[stream] = h.cam[0];
    t->cams[(size_t)t->B + stream] = h.cam[1];
    t->cam_dirty = true;
    return DVFE_OK;
}
}  // namespace

extern "C" int dvfe_export_stream(dvfe_tracker* t, int stream, void* blob, size_t cap, size_t* n_bytes) {
    if (!t || !n_bytes) { dvfe_set_error("export_stream: null argument"); return DVFE_ERR_INVALID; }
    if (!t->groups.empty()) {
        dvfe_tracker* leaf; int local;
        DVFE_CHECK(grp_route(t, stream, &leaf, &local));
        return dvfe_export_stream(leaf, local, blob, cap, n_bytes);
    }
    if (stream < 0 || stream >= t->B) { dvfe_set_error("export_stream: bad stream index %d", stream); return DVFE_ERR_INVALID; }
    return leaf_export(t, stream, static_cast<uint8_t*>(blob), cap, n_bytes);
}

extern "C" int dvfe_import_stream(dvfe_tracker* t, int stream, const void* blob, size_t n_bytes) {
    if (!t || !blob) { dvfe_set_error("import_stream: null argument"); return DVFE_ERR_INVALID; }
    if (!t->groups.empty()) {
        dvfe_tracker* leaf; int local;
        DVFE_CHECK(grp_route(t, stream, &leaf, &local));
        return dvfe_import_stream(leaf, local, blob, n_bytes);
    }
    if (stream < 0 || stream >= t->B) { dvfe_set_error("import_stream: bad stream index %d", stream); return DVFE_ERR_INVALID; }
    return leaf_import(t, stream, static_cast<const uint8_t*>(blob), n_bytes);
}
