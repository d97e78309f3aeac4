// Stream groups (dvfe_config::n_groups > 1): a container tracker that splits its B streams into G leaf trackers, each
// with its own compute / upload / download streams.  Streams are independent (SURVEY.md §8e), so the split changes
// nothing in the results; it lets the GPU overlap one group's latency-bound phases (one-CTA-per-stream corner
// selection, small bookkeeping kernels, launch tails) with another group's LK / response kernels.
#include <string.h>

#include "kernels.cuh"
#include "state.cuh"
#include "tracker.h"

#define DVFE_CHECK(call)                 \
    do {                                 \
        int rc__ = (call);               \
        if (rc__ != DVFE_OK) return rc__; \
    } while (0)

int grp_create(const dvfe_config* cfg, dvfe_tracker** out) {
    const int G = cfg->n_groups < cfg->n_streams ? cfg->n_groups : cfg->n_streams;
    dvfe_tracker* t = new dvfe_tracker();
    t->cfg = *cfg;
    t->B = cfg->n_streams; t->W = cfg->width; t->H = cfg->height; t->cap = cfg->max_cnt;
    t->group_first.push_back(0);
    for (int g = 0; g < G; g++) {
        dvfe_config c = *cfg;
        c.n_groups = 1;
        c.n_streams = cfg->n_streams / G + (g < cfg->n_streams % G ? 1 : 0);
        dvfe_tracker* leaf = nullptr;
        const int rc = dvfe_create(&c, &leaf);
        if (rc != DVFE_OK) {                       // keep the leaf's error message; release what was built
            for (dvfe_tracker* l : t->groups) dvfe_destroy(l);
            delete t;
            return rc;
        }
        t->groups.push_back(leaf);
        t->group_first.push_back(t->group_first.back() + c.n_streams);
    }
    *out = t;
    return DVFE_OK;
}

void grp_destroy(dvfe_tracker* t) {
    for (dvfe_tracker* g : t->groups) dvfe_destroy(g);
    delete t;
}

static int grp_of(const dvfe_tracker* t, int stream, int* local) {
    for (size_t g = 0; g + 1 < t->group_first.size(); g++)
        if (stream >= t->group_first[g] && stream < t->group_first[g + 1]) { *local = stream - t->group_first[g]; return (int)g; }
    return -1;
}

// every group submits a step, also one whose streams are all skipped, so that each dvfe_wait still pairs with one step per group
int grp_track_image_ex(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, size_t stride, int pitch,
                       const double* time0, const uint8_t* stream_flags, bool device) {
    for (size_t g = 0; g < t->groups.size(); g++) {
        const int f = t->group_first[g];
        const size_t off = (size_t)f * stride;
        DVFE_CHECK(dvfe_track_image_ex(t->groups[g], left + off, right ? right + off : nullptr, stride, pitch, time0 + f,
                                       stream_flags ? stream_flags + f : nullptr, device ? DVFE_STEP_DEVICE_INPUT : 0u));
    }
    return DVFE_OK;
}

int grp_wait(dvfe_tracker* t) {
    for (dvfe_tracker* g : t->groups) DVFE_CHECK(dvfe_wait(g));
    return DVFE_OK;
}

int grp_wait_all(dvfe_tracker* t) {
    for (dvfe_tracker* g : t->groups) DVFE_CHECK(g->wait_all());
    return DVFE_OK;
}

int grp_track_semantic(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, const uint8_t* inv, size_t stride, int pitch,
                       const int* exist, const double* time0, const uint8_t* stream_flags, unsigned flags) {
    for (size_t g = 0; g < t->groups.size(); g++) {
        const int f = t->group_first[g];
        const size_t off = (size_t)f * stride;
        const size_t moff = off / (size_t)(t->groups[g]->prep_active() ? t->groups[g]->in_ch : 1);
        DVFE_CHECK(dvfe_track_semantic_ex(t->groups[g], left + off, right ? right + off : nullptr, inv ? inv + moff : nullptr,
                                          stride, pitch, exist + f, time0 + f, stream_flags ? stream_flags + f : nullptr, flags));
    }
    return DVFE_OK;
}

int grp_insts_track(dvfe_tracker* t, int stream, const dvfe_inst_in* boxes, int n, double time0) {
    int local = 0;
    const int g = grp_of(t, stream, &local);
    if (g < 0) { dvfe_set_error("insts_track: bad stream"); return DVFE_ERR_INVALID; }
    return dvfe_insts_track(t->groups[g], local, boxes, n, time0);
}

int grp_insts_track_batch(dvfe_tracker* t, const dvfe_inst_in* boxes, const int* n_boxes, const double* time0) {
    size_t off = 0;
    for (size_t g = 0; g < t->groups.size(); g++) {
        const int f = t->group_first[g];
        DVFE_CHECK(dvfe_insts_track_batch(t->groups[g], boxes ? boxes + off : nullptr, n_boxes + f, time0 + f));
        for (int s = f; s < t->group_first[g + 1]; s++) off += (size_t)n_boxes[s];
    }
    return DVFE_OK;
}

// as grp_track_image_ex: every group submits a step, also one whose streams are all skipped
int grp_track_dynamic_async(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, const uint8_t* inv, size_t stride,
                            int pitch, const int* exist, const dvfe_inst_in* boxes, const int* n_boxes, const double* time0,
                            const uint8_t* stream_flags, unsigned flags) {
    size_t boff = 0;
    for (size_t g = 0; g < t->groups.size(); g++) {
        const int f = t->group_first[g];
        const size_t off = (size_t)f * stride;
        const size_t moff = off / (size_t)(t->groups[g]->prep_active() ? t->groups[g]->in_ch : 1);
        DVFE_CHECK(dvfe_track_dynamic_ex2(t->groups[g], left + off, right ? right + off : nullptr, inv ? inv + moff : nullptr,
                                          stride, pitch, exist ? exist + f : nullptr, boxes ? boxes + boff : nullptr, n_boxes + f,
                                          time0 + f, stream_flags ? stream_flags + f : nullptr, flags));
        for (int s = f; s < t->group_first[g + 1]; s++) boff += (size_t)n_boxes[s];
    }
    return DVFE_OK;
}

int grp_route(dvfe_tracker* t, int stream, dvfe_tracker** leaf, int* local) {
    const int g = t ? grp_of(t, stream, local) : -1;
    if (g < 0) { dvfe_set_error("bad stream index %d", stream); return DVFE_ERR_INVALID; }
    *leaf = t->groups[g];
    return DVFE_OK;
}

int grp_set_input(dvfe_tracker* t, int channels) {
    for (dvfe_tracker* g : t->groups) DVFE_CHECK(dvfe_set_input(g, channels));
    return DVFE_OK;
}

int grp_set_maps(dvfe_tracker* t, int cam, const int16_t* map1, const uint16_t* map2) {
    for (dvfe_tracker* g : t->groups) DVFE_CHECK(dvfe_set_undistort_maps(g, cam, map1, map2));
    return DVFE_OK;
}

int grp_set_stream_camera(dvfe_tracker* t, int stream, const dvfe_camera* cam0, const dvfe_camera* cam1) {
    dvfe_tracker* leaf; int local;
    DVFE_CHECK(grp_route(t, stream, &leaf, &local));
    return dvfe_set_stream_camera(leaf, local, cam0, cam1);
}

int grp_set_stream_maps(dvfe_tracker* t, int stream, int cam, const int16_t* map1, const uint16_t* map2) {
    dvfe_tracker* leaf; int local;
    DVFE_CHECK(grp_route(t, stream, &leaf, &local));
    return dvfe_set_stream_undistort_maps(leaf, local, cam, map1, map2);
}

int grp_set_lk_mode(dvfe_tracker* t, int site, int back_max_level, double fb) {
    for (dvfe_tracker* g : t->groups) DVFE_CHECK(dvfe_set_lk_mode_site(g, site, back_max_level, fb));
    return DVFE_OK;
}

int grp_set_detect_mode(dvfe_tracker* t, int mode) {
    for (dvfe_tracker* g : t->groups) DVFE_CHECK(dvfe_set_detect_mode(g, mode));
    return DVFE_OK;
}

int grp_set_reject_with_f(dvfe_tracker* t, double f_threshold) {
    for (dvfe_tracker* g : t->groups) DVFE_CHECK(dvfe_set_reject_with_f(g, f_threshold));
    return DVFE_OK;
}

int grp_profile(dvfe_tracker* t, int enable) {
    for (dvfe_tracker* g : t->groups) DVFE_CHECK(dvfe_profile(g, enable));
    return DVFE_OK;
}

// stage times summed over the groups (GPU time attributable to a stage per whole-tracker step; with overlapping
// groups the sum exceeds the wall time of the step)
int grp_profile_read(dvfe_tracker* t, const char** names, double* total_ms, long* steps) {
    double acc[16] = {0};
    int n = 0;
    long st = 0;
    for (dvfe_tracker* g : t->groups) {
        double ms[16];
        long s = 0;
        n = dvfe_profile_read(g, names, ms, &s);
        if (n < 0) return n;
        for (int i = 0; i < n; i++) acc[i] += ms[i];
        st = s;
    }
    if (total_ms) for (int i = 0; i < n; i++) total_ms[i] = acc[i];
    if (steps) *steps = st;
    return n;
}
