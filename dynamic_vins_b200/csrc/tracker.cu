// C ABI of libdvfe (include/dvfe.h): the batched, device-resident frame step that replaces
// FeatureTracker::TrackImage / TrackSemanticImage (dynamic_vins/src/front_end/background_tracker.cpp:52-158,
// 757-837) and the seam-level operators.  Host code only orchestrates launches; no pixel or point
// arithmetic happens on the CPU and there is no fallback when no CUDA device is present.
#include <limits.h>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "kernels.cuh"
#include "state.cuh"
#include "tracker.h"

unsigned long long g_dvfe_launches = 0;
static thread_local char g_err[512] = "";       // per calling thread: trackers on different host threads do not clobber each other

void dvfe_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

#define DVFE_CHECK(call)                 \
    do {                                 \
        int rc__ = (call);               \
        if (rc__ != DVFE_OK) return rc__; \
    } while (0)

// groups.cu
int grp_create(const dvfe_config* cfg, dvfe_tracker** out);
void grp_destroy(dvfe_tracker* t);
int grp_track_image_ex(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, size_t stride, int pitch,
                       const double* time0, const uint8_t* stream_flags, bool device);
int grp_wait(dvfe_tracker* t);
int grp_wait_all(dvfe_tracker* t);
int grp_track_semantic(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, const uint8_t* inv, size_t stride, int pitch,
                       const int* exist, const double* time0, const uint8_t* stream_flags, unsigned flags);
int grp_route(dvfe_tracker* t, int stream, dvfe_tracker** leaf, int* local);
int grp_set_lk_mode(dvfe_tracker* t, int site, int back_max_level, double fb);
int grp_set_detect_mode(dvfe_tracker* t, int mode);
int grp_set_reject_with_f(dvfe_tracker* t, double f_threshold);
int grp_profile(dvfe_tracker* t, int enable);
int grp_profile_read(dvfe_tracker* t, const char** names, double* total_ms, long* steps);
#define IS_GROUP(t) ((t) != nullptr && !(t)->groups.empty())

template <typename T>
static int dmalloc(T** p, size_t count) {
    DVFE_CUDA(cudaMalloc((void**)p, count * sizeof(T)));
    DVFE_CUDA(cudaMemset(*p, 0, count * sizeof(T)));
    return DVFE_OK;
}

// ---------------------------------------------------------------------------------------------------
int alloc_point_sets(PointSetArrays* S, int n_sets, int cap) {
    const size_t N = (size_t)n_sets * cap;
    DVFE_CHECK(dmalloc(&S->pts, N));
    DVFE_CHECK(dmalloc(&S->lk_out, N));
    DVFE_CHECK(dmalloc(&S->un, N));
    DVFE_CHECK(dmalloc(&S->vel, N));
    DVFE_CHECK(dmalloc(&S->ids, N));
    DVFE_CHECK(dmalloc(&S->track_cnt, N));
    DVFE_CHECK(dmalloc(&S->status, N));
    DVFE_CHECK(dmalloc(&S->rpts, N));
    DVFE_CHECK(dmalloc(&S->rstatus, N));
    DVFE_CHECK(dmalloc(&S->rprev_un, N));
    DVFE_CHECK(dmalloc(&S->rprev_valid, N));
    DVFE_CHECK(dmalloc(&S->n, (size_t)n_sets));
    return DVFE_OK;
}

void free_point_sets(PointSetArrays* S) {
    cudaFree(S->pts); cudaFree(S->lk_out); cudaFree(S->un); cudaFree(S->vel); cudaFree(S->ids);
    cudaFree(S->track_cnt); cudaFree(S->status); cudaFree(S->rpts); cudaFree(S->rstatus);
    cudaFree(S->rprev_un); cudaFree(S->rprev_valid); cudaFree(S->n);
    memset(S, 0, sizeof(*S));
}

int gftt_cells(int w, int h, float min_dist) {
    int cell = (int)lrintf(min_dist);
    if (cell < 1) cell = 1;
    return ((w + cell - 1) / cell) * ((h + cell - 1) / cell);
}

int alloc_gftt_scratch(GfttScratch* sc, int n_jobs, int w, int h, float min_dist) {
    sc->n_jobs = n_jobs;
    sc->w = w; sc->h = h;
    sc->mask_pitch = (w + 15) & ~15;
    sc->cand_cap = (w * h) / 4 + 4096;
    sc->n_cells = gftt_cells(w, h, min_dist);
    DVFE_CHECK(dmalloc(&sc->mask, (size_t)n_jobs * sc->mask_pitch * h));
    DVFE_CHECK(dmalloc(&sc->cand, (size_t)n_jobs * sc->cand_cap));
    DVFE_CHECK(dmalloc(&sc->cand2, (size_t)n_jobs * sc->cand_cap));
    DVFE_CHECK(dmalloc(&sc->cand3, (size_t)n_jobs * sc->cand_cap));
    DVFE_CHECK(dmalloc(&sc->state, (size_t)n_jobs * sc->cand_cap));
    DVFE_CHECK(dmalloc(&sc->cell_count, (size_t)n_jobs * 2 * (sc->n_cells + 1)));
    DVFE_CHECK(dmalloc(&sc->counters, (size_t)n_jobs * 8));
    {
        // counters 0..2 (n_precand, masked max as an ordered int, overflow) start reset; the selection kernel re-arms them
        std::vector<int> init((size_t)n_jobs * 8, 0);
        for (int j = 0; j < n_jobs; j++) init[(size_t)j * 8 + 1] = INT_MIN;
        DVFE_CUDA(cudaMemcpy(sc->counters, init.data(), init.size() * sizeof(int), cudaMemcpyHostToDevice));
    }
    return DVFE_OK;
}

void free_gftt_scratch(GfttScratch* sc) {
    cudaFree(sc->mask); cudaFree(sc->cand); cudaFree(sc->cand2); cudaFree(sc->cand3); cudaFree(sc->state);
    cudaFree(sc->cell_count); cudaFree(sc->counters);
    memset(sc, 0, sizeof(*sc));
}

void gftt_job_bind_scratch(GfttJob* J, const GfttScratch& sc, int j) {
    J->mask = sc.mask + (size_t)j * sc.mask_pitch * sc.h;
    J->mask_pitch = sc.mask_pitch;
    J->eig = nullptr;
    J->cand = sc.cand + (size_t)j * sc.cand_cap;
    J->cand2 = sc.cand2 + (size_t)j * sc.cand_cap;
    J->cand3 = sc.cand3 + (size_t)j * sc.cand_cap;
    J->cand_cap = sc.cand_cap;
    J->state = sc.state + (size_t)j * sc.cand_cap;
    J->cell_count = sc.cell_count + (size_t)j * 2 * (sc.n_cells + 1);
    J->counters = sc.counters + (size_t)j * 8;
}

static int check_device(int device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0) {
        dvfe_set_error("no CUDA device available (%s): libdvfe has no CPU fallback", cudaGetErrorString(e));
        return DVFE_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= count) {
        dvfe_set_error("device ordinal %d out of range (%d devices)", device, count);
        return DVFE_ERR_NO_DEVICE;
    }
    DVFE_CUDA(cudaSetDevice(device));
    return DVFE_OK;
}

// ---------------------------------------------------------------------------------------------------
extern "C" const char* dvfe_version(void) { return "dvfe 0.1 (sm_100a)"; }
extern "C" unsigned long long dvfe_kernel_launches(void) { return g_dvfe_launches; }
extern "C" const char* dvfe_last_error(const dvfe_tracker* t) { (void)t; return g_err; }

extern "C" int dvfe_create(const dvfe_config* cfg, dvfe_tracker** out) {
    if (!cfg || !out) { dvfe_set_error("dvfe_create: null argument"); return DVFE_ERR_INVALID; }
    *out = nullptr;
    if (cfg->width < 32 || cfg->height < 32 || cfg->n_streams < 1 || cfg->max_cnt < 1 || cfg->max_cnt > 2048 ||
        cfg->min_dist < 1 || cfg->lk_max_level < 0 || cfg->lk_max_level >= DVFE_MAX_PYR_LEVELS) {
        dvfe_set_error("dvfe_create: invalid config (w=%d h=%d streams=%d max_cnt=%d min_dist=%d lk_max_level=%d)",
                       cfg->width, cfg->height, cfg->n_streams, cfg->max_cnt, cfg->min_dist, cfg->lk_max_level);
        return DVFE_ERR_CONFIG;
    }
    DVFE_CHECK(check_device(cfg->device));
    if (cfg->n_groups > 1 && cfg->n_streams > 1) return grp_create(cfg, out);
    dvfe_tracker* t = new (std::nothrow) dvfe_tracker();
    if (!t) return DVFE_ERR_CAPACITY;
    t->cfg = *cfg;
    t->B = cfg->n_streams; t->W = cfg->width; t->H = cfg->height; t->cap = cfg->max_cnt;
    // levels for the forward maxLevel, the backward call's maxLevel 1 and the cv::cuda call pattern's 3 (dvfe_set_lk_mode)
    t->desc = make_pyr_desc(t->W, t->H, cfg->lk_max_level > 3 ? cfg->lk_max_level : 3);
    t->cams.assign((size_t)2 * t->B, make_cam(cfg->cam0));          // every stream with the config's cameras
    for (int s = 0; s < t->B; s++) t->cams[(size_t)t->B + s] = make_cam(cfg->cam1);
    int rc = t->init();
    if (rc != DVFE_OK) { dvfe_destroy(t); return rc; }
    *out = t;
    return DVFE_OK;
}

int dvfe_tracker::init() {
    DVFE_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    DVFE_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
    DVFE_CUDA(cudaStreamCreateWithFlags(&ds, cudaStreamNonBlocking));
    DVFE_CUDA(cudaStreamCreateWithFlags(&rs, cudaStreamNonBlocking));
    for (int p = 0; p < 2; p++) {
        for (int i = 0; i <= ST_COUNT; i++) DVFE_CUDA(cudaEventCreate(&ev[p][i]));
        DVFE_CUDA(cudaEventCreateWithFlags(&ev_up[p], cudaEventDisableTiming));
        DVFE_CUDA(cudaEventCreateWithFlags(&ev_packed[p], cudaEventDisableTiming));
        DVFE_CUDA(cudaEventCreateWithFlags(&ev_resp[p], cudaEventDisableTiming));
        DVFE_CUDA(cudaEventCreateWithFlags(&ev_rpyr[p], cudaEventDisableTiming));
        DVFE_CUDA(cudaEventCreateWithFlags(&ev_r0[p], cudaEventDisableTiming));
        DVFE_CUDA(cudaEventCreateWithFlags(&ev_begin[p], cudaEventDisableTiming));
        DVFE_CUDA(cudaEventCreateWithFlags(&ev_done[p], cudaEventDisableTiming));
    }
    const size_t P = (size_t)W * H;
    for (int s = 0; s < 3; s++) DVFE_CHECK(dmalloc(&pyrL[s], (size_t)B * desc.bytes));
    for (int s = 0; s < 2; s++) DVFE_CHECK(dmalloc(&pyrR[s], (size_t)B * desc.bytes));
    DVFE_CHECK(alloc_point_sets(&bg, B, cap));
    DVFE_CHECK(dmalloc(&d_next_id, (size_t)B));
    {
        std::vector<uint32_t> ones(B, 1u);     // InstFeat::global_id_count{1}
        DVFE_CUDA(cudaMemcpy(d_next_id, ones.data(), B * sizeof(uint32_t), cudaMemcpyHostToDevice));
    }
    DVFE_CHECK(dmalloc(&d_dt, (size_t)B));
    DVFE_CHECK(dmalloc(&d_err, (size_t)2));
    prev_time.assign(B, 0.0);
    tc_valid.assign(B, 0);
    last_sflags.assign(B, 0);
    had_frame.assign(B, 0);
    DVFE_CHECK(dmalloc(&d_sflags, (size_t)B));
    DVFE_CHECK(dmalloc(&d_lane, (size_t)B));
    DVFE_CHECK(dmalloc(&d_pgroups[0], (size_t)B));
    DVFE_CHECK(dmalloc(&d_pgroups[1], (size_t)B));
    DVFE_CHECK(dmalloc(&d_pjobs, (size_t)B));
    DVFE_CHECK(dmalloc(&d_zero, (size_t)1));
    DVFE_CHECK(dmalloc(&d_cam, cams.size()));
    DVFE_CUDA(cudaMemcpy(d_cam, cams.data(), cams.size() * sizeof(CamParams), cudaMemcpyHostToDevice));
    for (int p = 0; p < 2; p++) DVFE_CUDA(cudaMallocHost((void**)&h_cam[p], cams.size() * sizeof(CamParams)));
    for (int cam = 0; cam < 2; cam++) {
        own_maps[cam].assign(B, 0);
        s_map1[cam].assign(B, nullptr);
        s_map2[cam].assign(B, nullptr);
        DVFE_CHECK(dmalloc(&d_imaps[cam], (size_t)B));          // all null: no maps
    }
    for (int p = 0; p < 2; p++) {
        DVFE_CUDA(cudaMallocHost((void**)&h_sflags[p], (size_t)B));
        memset(h_sflags[p], 0, (size_t)B);
    }
    DVFE_CHECK(dmalloc(&d_src, (size_t)3 * B));
    for (int p = 0; p < 2; p++) DVFE_CUDA(cudaMallocHost((void**)&h_src[p], (size_t)3 * B * sizeof(ImgSrc)));
    for (int p = 0; p < 2; p++) {
        DVFE_CHECK(dmalloc(&d_obs[p], (size_t)B * 2 * cap));
        DVFE_CHECK(dmalloc(&d_nobs[p], (size_t)B));
        DVFE_CUDA(cudaMallocHost((void**)&h_dt[p], B * sizeof(double)));
        DVFE_CUDA(cudaMallocHost((void**)&h_obs[p], (size_t)B * 2 * cap * sizeof(dvfe_obs)));
        DVFE_CUDA(cudaMallocHost((void**)&h_nobs[p], (B + 1) * sizeof(int)));
        memset(h_nobs[p], 0, (B + 1) * sizeof(int));
    }
    DVFE_CHECK(dmalloc(&d_region, (size_t)B * P));
    DVFE_CHECK(dmalloc(&d_region_tmp, (size_t)B * P));
    DVFE_CHECK(dmalloc(&d_exist, (size_t)B));
    for (int p = 0; p < 2; p++) {
        DVFE_CHECK(dmalloc(&d_inv_in[p], (size_t)B * P));
        DVFE_CUDA(cudaMallocHost((void**)&h_exist[p], B * sizeof(int)));
        DVFE_CUDA(cudaEventCreateWithFlags(&ev_inst[p], cudaEventDisableTiming));
    }
    DVFE_CHECK(alloc_gftt_scratch(&gsc, B, W, H, (float)cfg.min_dist));
    DVFE_CHECK(gftt_prepare_device());
    {
        // level 0 of every stream of a left slot as one 2-D byte tensor: a pyramid is a whole number of level-0 rows
        const PyrLevel& L0 = desc.lv[0];
        const long rows = (long)B * (long)(desc.bytes / (unsigned)L0.pitch);
        use_tma = true;
        for (int s = 0; s < 3 && use_tma; s++)
            use_tma = dvfe_make_level0_tmap(tmapL[s], pyrL[s] + L0.offset, L0.pitch, rows) == DVFE_OK;
        if (const char* e = getenv("DVFE_TMA")) use_tma = use_tma && atoi(e) != 0;          // A/B: 0 = cp.async staging
    }
    // pitched host->device DMA straight into the padded level 0 runs at full PCIe rate only for rows that are a
    // multiple of 64 bytes; other widths go through a dense staging buffer (one linear copy) and the copy kernel
    staged_upload = (W % 64) != 0;
    if (const char* e = getenv("DVFE_GRAPHS")) use_graphs = atoi(e) != 0;                // A/B: 0 = plain launches
    if (const char* e = getenv("DVFE_REUSE")) use_reuse = atoi(e) != 0;
    DVFE_CHECK(size_stage());

    if (cfg.stereo) {
        DVFE_CHECK(dmalloc(&d_tcache, (size_t)B * cap * DVFE_MAX_PYR_LEVELS * LK_TCACHE_WORDS));
        DVFE_CHECK(dmalloc(&d_tcache_bwd, (size_t)B * cap * DVFE_MAX_PYR_LEVELS * LK_TCACHE_WORDS));
        DVFE_CHECK(dmalloc(&d_old_idx, (size_t)B * cap));
    }
    // LK groups: [phase][temporal raw | temporal semantic | stereo]
    std::vector<LkGroup> g(B);
    for (int ph = 0; ph < 6; ph++) {
        uint8_t* cur = left_slot(ph);
        uint8_t* prev = left_slot(ph + 2);
        for (int kind = 0; kind < 3; kind++) {
            for (int s = 0; s < B; s++) {
                LkGroup& G = g[s];
                memset(&G, 0, sizeof(G));
                G.desc = desc;
                const size_t o = (size_t)s * cap;
                if (kind < 2) {
                    G.pyrA = prev + (size_t)s * desc.bytes;
                    G.pyrB = cur + (size_t)s * desc.bytes;
                    G.ptsA = bg.pts + o; G.ptsB = bg.lk_out + o; G.status = bg.status + o;
                    if (kind == 1) { G.mask = d_region + (size_t)s * P; G.mask_pitch = W; }
                } else {
                    G.pyrA = cur + (size_t)s * desc.bytes;
                    G.pyrB = right_slot(ph) + (size_t)s * desc.bytes;
                    G.ptsA = bg.pts + o; G.ptsB = bg.rpts + o; G.status = bg.rstatus + o;
                }
                G.n = bg.n + s;
                G.tcache = d_tcache ? d_tcache + (size_t)s * cap * DVFE_MAX_PYR_LEVELS * LK_TCACHE_WORDS : nullptr;
                G.tcache_bwd = d_tcache_bwd ? d_tcache_bwd + (size_t)s * cap * DVFE_MAX_PYR_LEVELS * LK_TCACHE_WORDS : nullptr;
                G.old_idx = d_old_idx ? d_old_idx + o : nullptr;
            }
            DVFE_CHECK(dmalloc(&d_groups[ph][kind], (size_t)B));
            DVFE_CUDA(cudaMemcpy(d_groups[ph][kind], g.data(), B * sizeof(LkGroup), cudaMemcpyHostToDevice));
        }
    }
    // GFTT jobs: [phase][raw | semantic | semantic with the cv::cuda detector's threshold (TrackImageNaive)]
    std::vector<GfttJob> jobs(B);
    for (int ph = 0; ph < 6; ph++)
        for (int kind = 0; kind < 3; kind++) {
            for (int s = 0; s < B; s++) {
                GfttJob& J = jobs[s];
                memset(&J, 0, sizeof(J));
                const PyrLevel& L0 = desc.lv[0];
                J.img = left_slot(ph) + (size_t)s * desc.bytes + L0.offset + (size_t)DVFE_PADY * L0.pitch + DVFE_PADX;
                J.img_pitch = L0.pitch;
                J.w = W; J.h = H;
                J.img_bordered = 1;
                if (kind >= 1) { J.region_mask = d_region + (size_t)s * P; J.region_pitch = W; }
                J.max_unmasked = kind == 2 ? 1 : 0;
                gftt_job_bind_scratch(&J, gsc, s);
                const size_t o = (size_t)s * cap;
                J.pts = bg.pts + o; J.ids = bg.ids + o; J.track_cnt = bg.track_cnt + o;
                J.n = bg.n + s; J.next_id = d_next_id + s;
                J.max_cnt = cfg.max_cnt;
                J.min_needed = kind == 0 ? 1 : 10;    // TrackImage: n_max_cnt > 0; DetectNewFeature: n_max_cnt >= 10
                J.disc_radius = cfg.min_dist;
                J.min_dist = (float)cfg.min_dist;
                J.quality = 0.01;
                J.err = d_err + (ph % 2);       // the error word of the step this job table belongs to
            }
            DVFE_CHECK(dmalloc(&d_jobs[ph][kind], (size_t)B));
            DVFE_CUDA(cudaMemcpy(d_jobs[ph][kind], jobs.data(), B * sizeof(GfttJob), cudaMemcpyHostToDevice));
        }
    DVFE_CHECK(init_instances());
    DVFE_CUDA(cudaDeviceSynchronize());
    return DVFE_OK;
}

extern "C" void dvfe_destroy(dvfe_tracker* t) {
    if (!t) return;
    if (IS_GROUP(t)) { grp_destroy(t); return; }
    cudaSetDevice(t->cfg.device);
    if (t->st) cudaStreamSynchronize(t->st);
    if (t->cs) cudaStreamSynchronize(t->cs);
    if (t->ds) cudaStreamSynchronize(t->ds);
    if (t->rs) cudaStreamSynchronize(t->rs);
    t->drop_graphs();
    for (int s = 0; s < 3; s++) cudaFree(t->pyrL[s]);
    for (int s = 0; s < 2; s++) cudaFree(t->pyrR[s]);
    free_point_sets(&t->bg);
    cudaFree(t->d_next_id); cudaFree(t->d_dt); cudaFree(t->d_err); cudaFree(t->d_tcache); cudaFree(t->d_tcache_bwd);
    cudaFree(t->d_old_idx); cudaFree(t->d_fm_models);
    cudaFree(t->d_sflags); cudaFree(t->d_lane); cudaFree(t->d_pgroups[0]); cudaFree(t->d_pgroups[1]); cudaFree(t->d_pjobs);
    cudaFree(t->d_zero);
    cudaFree(t->d_src);
    cudaFree(t->d_cam);
    cudaFree(t->d_snap);
    for (int cam = 0; cam < 2; cam++) {
        cudaFree(t->d_imaps[cam]);
        for (short* m : t->s_map1[cam]) cudaFree(m);
        for (unsigned short* m : t->s_map2[cam]) cudaFree(m);
    }
    for (int p = 0; p < 2; p++) {
        cudaFreeHost(t->h_sflags[p]);
        cudaFreeHost(t->h_src[p]);
        cudaFreeHost(t->h_cam[p]);
        cudaFree(t->d_obs[p]); cudaFree(t->d_nobs[p]);
        if (t->ev_packed[p]) cudaEventDestroy(t->ev_packed[p]);
        if (t->ev_resp[p]) cudaEventDestroy(t->ev_resp[p]);
        if (t->ev_rpyr[p]) cudaEventDestroy(t->ev_rpyr[p]);
        if (t->ev_r0[p]) cudaEventDestroy(t->ev_r0[p]);
        if (t->ev_begin[p]) cudaEventDestroy(t->ev_begin[p]);
        cudaFreeHost(t->h_dt[p]); cudaFreeHost(t->h_obs[p]); cudaFreeHost(t->h_nobs[p]);
        if (t->ev_up[p]) cudaEventDestroy(t->ev_up[p]);
        if (t->ev_done[p]) cudaEventDestroy(t->ev_done[p]);
        for (int i = 0; i <= dvfe_tracker::ST_COUNT; i++) if (t->ev[p][i]) cudaEventDestroy(t->ev[p][i]);
    }
    for (int i = 0; i < 2; i++) { cudaFree(t->d_stage[i]); cudaFree(t->d_map1[i]); cudaFree(t->d_map2[i]); }
    cudaFree(t->d_region); cudaFree(t->d_region_tmp); cudaFree(t->d_exist);
    for (int p = 0; p < 2; p++) {
        cudaFree(t->d_labels[p]);
        cudaFree(t->d_inv_in[p]); cudaFreeHost(t->h_exist[p]);
        if (t->ev_inst[p]) cudaEventDestroy(t->ev_inst[p]);
    }
    free_gftt_scratch(&t->gsc);
    for (int p = 0; p < 6; p++) {
        for (int k = 0; k < 3; k++) cudaFree(t->d_groups[p][k]);
        for (int k = 0; k < 3; k++) cudaFree(t->d_jobs[p][k]);
    }
    t->free_instances();
    if (t->cs) cudaStreamDestroy(t->cs);
    if (t->ds) cudaStreamDestroy(t->ds);
    if (t->rs) cudaStreamDestroy(t->rs);
    if (t->st && t->own_stream) cudaStreamDestroy(t->st);
    delete t;
}

// ---- the frame step --------------------------------------------------------------------------------------
// submit() only enqueues: optional device-side copy into level 0, pyramids, LK, detection, post-processing and the
// D2H of the records of step k, all on the compute stream; nothing blocks the host.  Two steps may be in flight,
// so the H2D of step k+1 (upload stream) overlaps the kernels of step k.
void dvfe_tracker::drop_graphs() {
    for (auto& kv : step_graphs)
        if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    step_graphs.clear();
}

// The kernels of one frame step on the compute stream `st` (+ the right pyramid on `rs`, forked and joined by events).
// No host-dependent state is read: the same call with the same arguments enqueues the same work, which is what lets
// submit() capture it into a graph.
// partial: a step with some stream flag set.  The same kernels run on the partial tables (presence.cu), which k_partial_tables
// derives from the flags copied here and the tables of this phase and mode; skipped streams' previous pyramids are carried.
int dvfe_tracker::enqueue_compute(const uint8_t* d_left, const uint8_t* d_right, size_t stream_stride, int pitch, bool semantic,
                                  int level0_mode, bool stereo_now, long k, bool with_marks, bool partial) {
    const int ph = (int)(k % 6), par = (int)(k % 2);
    auto mark = [&](int i) { if (with_marks) cudaEventRecord(ev[par][i], st); };
    DVFE_CUDA(cudaMemcpyAsync(d_dt, h_dt[par], B * sizeof(double), cudaMemcpyHostToDevice, st));
    // the capacity flag is per step: cleared here, reported by the wait for THIS step only (the buffers of step k-2 have
    // been read back before slot `par` is reused)
    DVFE_CUDA(cudaMemsetAsync(d_err + par, 0, sizeof(int), st));
    mark(0);
    // One set of partial tables serves every step: all their readers run on this stream, before the next step rebuilds them.
    if (partial) {
        DVFE_CUDA(cudaMemcpyAsync(d_sflags, h_sflags[par], (size_t)B, cudaMemcpyHostToDevice, st));
        PartialTables pt;
        pt.full_temporal = d_groups[ph][semantic ? 1 : 0]; pt.full_stereo = d_groups[ph][2];
        pt.full_jobs = d_jobs[ph][semantic ? (detect_cuda ? 2 : 1) : 0];
        pt.temporal = d_pgroups[0]; pt.stereo = d_pgroups[1]; pt.jobs = d_pjobs; pt.lane = d_lane;
        pt.zero = d_zero; pt.n = bg.n; pt.next_id = d_next_id;
        DVFE_CHECK(launch_partial_tables(pt, d_sflags, B, stereo_now ? 1 : 0, st));     // also RESET: n = 0, next_id = 1
    }
    const uint8_t* lane = partial ? d_lane : nullptr;
    // left pyramid now; the right pyramid is built on its own stream while the selection kernel (one CTA per
    // stream) leaves most SMs idle, and joins before the stereo LK
    PyrImgSet set;
    set.src[0] = d_left; set.src[1] = nullptr;
    set.dst[0] = left_slot(k); set.dst[1] = nullptr;
    set.src_stride = stream_stride; set.dst_stride = desc.bytes; set.per_set = B;
    DVFE_CHECK(launch_build_pyramids(set, B, desc, pitch, st, level0_mode));
    // A skipped stream's "current" pyramid becomes its previous one again.  Nothing else touches either slot meanwhile: the
    // upload of step k+1 writes slot (k+1) % 3, and the uploads (place_input, the device-input copy in submit) wait for step k-2,
    // the last reader of that slot, before they write it; slots k % 3 and (k+2) % 3 are read only by this step's kernels.
    if (partial) DVFE_CHECK(launch_carry_pyramids(left_slot(k), left_slot(k + 2), desc.bytes, d_sflags, B, st));
    mark(ST_PYRAMID + 1);
    // The temporal call's backward templates (current left image at the tracked positions, levels <= its backward maxLevel)
    // are the stereo call's forward templates at those levels for the survivors: stored by the former, picked up through
    // the compaction's old-index map by the latter.
    const int site_t = semantic ? DVFE_LK_SEMANTIC_TEMPORAL : DVFE_LK_RAW_TEMPORAL;
    const bool reuse = use_reuse && k > 0 && stereo_now && cfg.flow_back && d_tcache_bwd != nullptr;
    // in a partial step the table decides per stream whether its cache is read (tc_valid)
    const bool tc_read = partial ? d_tcache != nullptr : tcache_valid;
    if (k > 0)   // bg.TrackLeft / FeatureTrackByLK(prev.gray0, gray0, last_points)
        DVFE_CHECK(launch_lk(partial ? d_pgroups[0] : d_groups[ph][semantic ? 1 : 0], B, cap, cfg.lk_max_level, cfg.flow_back, st,
                             lk_back_level[site_t], lk_fb_thresh[site_t], (tc_read ? LK_TCACHE_READ : 0) | (reuse ? LK_TCACHE_WRITE_BWD : 0)));
    mark(ST_LK_TEMPORAL + 1);
    // RejectWithF (dvfe_set_reject_with_f): the survivors that fit no common epipolar geometry lose their status before the
    // compaction; timed with it (the "compact" stage)
    if (k > 0 && reject_f > 0.0)
        DVFE_CHECK(launch_reject_with_f_step(bg, B, cap, d_cam, lane, W, H, reject_f, d_fm_models, st));
    if (k > 0)   // ReduceVector x4 + track_cnt++
        DVFE_CHECK(launch_compact(bg, B, cap, st, lane, reuse ? d_old_idx : nullptr));
    mark(ST_COMPACT + 1);
    // discs + goodFeaturesToTrack + ids
    DVFE_CHECK(launch_gftt(partial ? d_pjobs : d_jobs[ph][semantic ? (detect_cuda ? 2 : 1) : 0], nullptr, B, W, H, cap, st, with_marks ? &ev[par][ST_GFTT_MASK + 1] : nullptr,
                           stereo_now ? ev_resp[par] : nullptr, use_tma ? tmapL[k % 3] : nullptr,
                           (int)(desc.bytes / (unsigned)desc.lv[0].pitch)));
    if (stereo_now) {
        PyrImgSet rset;
        rset.src[0] = d_right; rset.src[1] = nullptr;
        rset.dst[0] = right_slot(k); rset.dst[1] = nullptr;
        rset.src_stride = stream_stride; rset.dst_stride = desc.bytes; rset.per_set = B;
        DVFE_CUDA(cudaStreamWaitEvent(rs, ev_resp[par], 0));        // after the response kernel of this step (and so
        DVFE_CHECK(launch_build_pyramids(rset, B, desc, pitch, rs, level0_mode));   // after the upload it waited for)
        DVFE_CUDA(cudaEventRecord(ev_rpyr[par], rs));
    }
    mark(ST_GFTT_SELECT + 1);
    // UndistortedPts(cam0) + PtsVelocity, each stream with its own cam0
    DVFE_CHECK(launch_left_post(bg, B, cap, d_cam, 1, d_dt, nullptr, st, lane));
    mark(ST_LEFT_POST + 1);
    if (stereo_now) DVFE_CUDA(cudaStreamWaitEvent(st, ev_rpyr[par], 0));
    if (stereo_now)   // FeatureTrackByLK(gray0, gray1, curr_points) — left points are kept when the match fails
        DVFE_CHECK(launch_lk(partial ? d_pgroups[1] : d_groups[ph][2], B, cap, cfg.lk_max_level, cfg.flow_back, st,
                             lk_back_level[semantic ? DVFE_LK_SEMANTIC_STEREO : DVFE_LK_RAW_STEREO],
                             lk_fb_thresh[semantic ? DVFE_LK_SEMANTIC_STEREO : DVFE_LK_RAW_STEREO],
                             LK_TCACHE_WRITE | (reuse ? LK_TCACHE_READ_BWD : 0), reuse ? lk_back_level[site_t] : -1));
    mark(ST_LK_STEREO + 1);
    DVFE_CHECK(launch_right_post_pack(bg, B, cap, d_cam + B, d_dt, stereo_now ? 1 : 0, d_obs[par], d_nobs[par], st, lane));
    mark(ST_PACK + 1);
    return DVFE_OK;
}

// Capture and instantiate the graph of the step with buffer phase `ph` and mode `flags` (bit 0 semantic, 2 stereo, 3 not the first
// frame, 4 forward templates cached, 5 level 0 arrives with its border, 6 partial: per-stream flags, bit 4 unused); `k` = any frame
// index with k % 6 == ph and (k > 0) as in the flags.  Nothing runs.
int dvfe_tracker::capture_step(int ph, unsigned flags, long k) {
    const unsigned long long before = g_dvfe_launches;
    const bool keep_valid = tcache_valid;
    tcache_valid = (flags & 16u) != 0;
    cudaGraph_t g = nullptr;
    DVFE_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
    const int rc = enqueue_compute(nullptr, nullptr, 0, 0, (flags & 1u) != 0, (flags & 32u) ? DVFE_L0_COMPLETE : DVFE_L0_INTERIOR,
                                   (flags & 4u) != 0, k, false, (flags & 64u) != 0);
    const cudaError_t ce = cudaStreamEndCapture(st, &g);
    tcache_valid = keep_valid;
    const unsigned n_kernels = (unsigned)(g_dvfe_launches - before);
    g_dvfe_launches = before;                              // nothing ran yet
    if (rc != DVFE_OK || ce != cudaSuccess) {
        if (g) cudaGraphDestroy(g);
        if (rc != DVFE_OK) return rc;
        dvfe_set_error("stream capture of the frame step failed: %s", cudaGetErrorString(ce));
        return DVFE_ERR_CUDA;
    }
    StepGraph sg;
    sg.n_kernels = n_kernels;
    const cudaError_t ie = cudaGraphInstantiate(&sg.exec, g, 0);
    cudaGraphDestroy(g);
    if (ie != cudaSuccess) { dvfe_set_error("cudaGraphInstantiate: %s", cudaGetErrorString(ie)); return DVFE_ERR_CUDA; }
    step_graphs.emplace(StepKey(ph, flags), sg);
    return DVFE_OK;
}

int dvfe_tracker::submit(const StepInput& in, const double* time0, bool semantic, const uint8_t* sflags) {
    const long k = frames;
    const int ph = (int)(k % 6), par = (int)(k % 2);
    const bool stereo_now = cfg.stereo && in.has_right;
    const bool partial = sflags != nullptr;
    // the frame index the compute part runs as: frame 6 has the buffer phase of frame 0 and is not a first frame (prev_loaded)
    const long kc = (k == 0 && prev_loaded) ? 6 : k;
    if (partial) {
        for (int s = 0; s < B; s++) {
            if (sflags[s] & DVFE_FRAME_RESET) prev_time[s] = 0.0;                  // a new tracker's prev_time
            h_dt[par][s] = (sflags[s] & DVFE_FRAME_SKIP) ? 0.0 : time0[s] - prev_time[s];
            h_sflags[par][s] = (uint8_t)(sflags[s] | (tc_valid[s] ? SF_TCACHE_VALID : 0u));
        }
    } else {
        for (int s = 0; s < B; s++) h_dt[par][s] = time0[s] - prev_time[s];       // cur_time - prev_time
    }
    prof_step[par] = prof;
    if (cam_dirty) {
        // the calibration of this step (dvfe_set_stream_camera), ahead of its kernels and behind those of every earlier step.
        // h_cam[par] was last the source of step k-2's copy, which has completed (wait_slot).
        memcpy(h_cam[par], cams.data(), cams.size() * sizeof(CamParams));
        DVFE_CUDA(cudaMemcpyAsync(d_cam, h_cam[par], cams.size() * sizeof(CamParams), cudaMemcpyHostToDevice, st));
        cam_dirty = false;
    }
    // everything step k-1 (background and instances) put on the compute stream lies before this point
    DVFE_CUDA(cudaEventRecord(ev_begin[par], st));
    if (use_graphs && !prof) {
        // The captured step never sees the caller's image pointers: device-resident input is copied into level 0 here,
        // left on the compute stream, right on its own stream behind the last readers of that slot (the stereo LKs of step
        // k-2, all of which precede the start of step k-1), and the graph runs as if level 0 had arrived in place.
        if (!in.in_place) {
            PyrImgSet set;
            set.src[0] = in.left; set.src[1] = nullptr; set.dst[0] = left_slot(k); set.dst[1] = nullptr;
            set.src_stride = in.stride; set.dst_stride = desc.bytes; set.per_set = B;
            DVFE_CHECK(launch_pyr_level0(set, B, desc, in.pitch, st));
            if (stereo_now) {
                set.src[0] = in.right; set.dst[0] = right_slot(k);
                if (k >= 1) DVFE_CUDA(cudaStreamWaitEvent(rs, ev_begin[1 - par], 0));
                // ... and behind the upload of this step when the source is the tracker's own staging buffer (widths whose rows
                // are not a multiple of 64 bytes); for caller-resident images the event is an old, completed one
                DVFE_CUDA(cudaStreamWaitEvent(rs, ev_up[par], 0));
                DVFE_CHECK(launch_pyr_level0(set, B, desc, in.pitch, rs));
                DVFE_CUDA(cudaEventRecord(ev_r0[par], rs));
                DVFE_CUDA(cudaStreamWaitEvent(st, ev_r0[par], 0));
            }
        }
        // level 0 copied by the kernel above (or by the gather form of it in place_table) arrives with its border; DMA / ingest
        // kernels leave the border to the graph
        const bool l0_complete = (!in.in_place && pyr_level0_writes_border(desc)) || in.l0_border;
        const unsigned flags = (semantic ? 1u : 0u) | (stereo_now ? 4u : 0u) | (kc > 0 ? 8u : 0u) | (tcache_valid && !partial ? 16u : 0u) |
                               (l0_complete ? 32u : 0u) | (partial ? 64u : 0u);
        const StepKey key(ph, flags);
        if (step_graphs.find(key) == step_graphs.end()) {
            if (step_graphs.size() >= 64) drop_graphs();          // a caller cycling through many modes
            DVFE_CHECK(capture_step(ph, flags, kc));
            // The first step of a mode also captures the six steady-state graphs it will replay from the next frame on (one per
            // buffer phase), so that instantiation (host time, ~0.3 ms each) never falls into a later, possibly timed, step.
            const bool tc_next = stereo_now && d_tcache != nullptr;
            const unsigned steady = (semantic ? 1u : 0u) | (stereo_now ? 4u : 0u) | 8u | (tc_next && !partial ? 16u : 0u) |
                                    (l0_complete ? 32u : 0u) | (partial ? 64u : 0u);
            for (int p = 0; p < 6; p++)
                if (step_graphs.find(StepKey(p, steady)) == step_graphs.end()) DVFE_CHECK(capture_step(p, steady, 6 + p));
        }
        auto it = step_graphs.find(key);
        DVFE_CUDA(cudaGraphLaunch(it->second.exec, st));
        g_dvfe_launches += it->second.n_kernels;
    } else {
        DVFE_CHECK(enqueue_compute(in.left, in.right, in.stride, in.pitch, semantic,
                                   in.in_place ? (in.l0_border ? DVFE_L0_COMPLETE : DVFE_L0_INTERIOR) : DVFE_L0_BUILD,
                                   stereo_now, kc, prof, partial));
    }
    // Template-cache validity per stream: a present frame with a stereo step leaves the templates of its points, a frame without
    // one leaves none (a RESET frame's points are all new), a skipped stream keeps what it had.  A full step reads the cache of
    // every stream or of none, so it reads it only when every stream's is valid.
    if (partial) {
        bool all = true;
        for (int s = 0; s < B; s++) {
            if (!(sflags[s] & DVFE_FRAME_SKIP)) tc_valid[s] = stereo_now && d_tcache != nullptr && !(sflags[s] & DVFE_FRAME_NO_RIGHT);
            all = all && tc_valid[s];
        }
        tcache_valid = all;
    } else {
        tcache_valid = stereo_now && d_tcache != nullptr;
        tc_valid.assign(B, tcache_valid ? 1 : 0);
    }
    // records go home on the download stream so that the next step's kernels do not queue behind the copy
    DVFE_CUDA(cudaEventRecord(ev_packed[par], st));
    DVFE_CUDA(cudaStreamWaitEvent(ds, ev_packed[par], 0));
    DVFE_CUDA(cudaMemcpyAsync(h_nobs[par], d_nobs[par], B * sizeof(int), cudaMemcpyDeviceToHost, ds));
    DVFE_CUDA(cudaMemcpyAsync(h_nobs[par] + B, d_err + par, sizeof(int), cudaMemcpyDeviceToHost, ds));
    DVFE_CUDA(cudaMemcpyAsync(h_obs[par], d_obs[par], (size_t)B * 2 * cap * sizeof(dvfe_obs), cudaMemcpyDeviceToHost, ds));
    if (prof) cudaEventRecord(ev[par][ST_D2H + 1], ds);
    DVFE_CUDA(cudaEventRecord(ev_done[par], ds));
    for (int s = 0; s < B; s++)
        if (!partial || !(sflags[s] & DVFE_FRAME_SKIP)) { prev_time[s] = time0[s]; had_frame[s] = 1; }
    last_has_right = stereo_now;
    if (partial) last_sflags.assign(sflags, sflags + B);
    else last_sflags.assign(B, 0);
    frames++;
    return DVFE_OK;
}

int dvfe_tracker::wait_one() {
    if (completed >= frames) return DVFE_OK;
    const int par = (int)(completed % 2);
    DVFE_CUDA(cudaEventSynchronize(ev_done[par]));
    if (prof_step[par]) {
        for (int i = 0; i < ST_COUNT; i++) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, ev[par][i], ev[par][i + 1]) == cudaSuccess) prof_ms[i] += ms;
        }
        prof_steps++;
    }
    out_slot = par;
    completed++;
    if (inst_pending[par]) {
        inst_pending[par] = false;
        DVFE_CUDA(cudaEventSynchronize(ev_inst[par]));
        DVFE_CHECK(finish_instances(par));
    }
    if (h_nobs[par][B] != 0) {
        dvfe_set_error("corner detection: more local maxima than the candidate buffer holds (W*H/4 + 4096); "
                       "the corner selection of this frame was truncated in at least one stream");
        return DVFE_ERR_CAPACITY;
    }
    return DVFE_OK;
}

int dvfe_tracker::wait_all() {
    while (completed < frames) DVFE_CHECK(wait_one());
    return DVFE_OK;
}

int dvfe_tracker::wait_slot() {
    while (frames - completed >= 2) DVFE_CHECK(wait_one());
    return DVFE_OK;
}

// ---- the step's input: host or device images -> where the step reads them ---------------------------------------------
uint8_t* dvfe_tracker::level0(int cam) const {
    const PyrLevel& L0 = desc.lv[0];
    return (cam ? right_slot(frames) : left_slot(frames)) + L0.offset + (size_t)DVFE_PADY * L0.pitch + DVFE_PADX;
}

// remap (if camera `cam` has maps) + gray conversion of B device images into level 0 of this step's pyramid slot: the
// shared-map kernel when every stream of the camera uses the same maps (or none), the per-image kernel otherwise
int dvfe_tracker::ingest(const uint8_t* d_src, size_t stream_stride, int pitch, int cam, cudaStream_t s) {
    IngestArgs a;
    a.src = d_src; a.src_stride = stream_stride; a.src_pitch = pitch; a.ch = in_ch;
    a.map1 = maps_uniform[cam] ? stream_map1(cam, 0) : nullptr;
    a.map2 = maps_uniform[cam] ? stream_map2(cam, 0) : nullptr;
    a.dst = level0(cam);
    a.dst_stride = desc.bytes; a.dst_pitch = desc.lv[0].pitch;
    a.w = W; a.h = H; a.n_img = B; a.keep_channels = 0;
    return launch_ingest(a, s, maps_uniform[cam] ? nullptr : d_imaps[cam]);
}

int dvfe_tracker::update_maps(int cam) {
    std::vector<IngestMaps> m(B);
    bool uniform = true;
    for (int s = 0; s < B; s++) {
        m[s].map1 = stream_map1(cam, s); m[s].map2 = stream_map2(cam, s);
        uniform = uniform && m[s].map1 == m[0].map1;
    }
    maps_uniform[cam] = uniform;
    DVFE_CUDA(cudaMemcpy(d_imaps[cam], m.data(), B * sizeof(IngestMaps), cudaMemcpyHostToDevice));
    return DVFE_OK;
}

// B host images of H rows of `row` bytes -> device memory, on the upload stream.  Into the dense staging: one linear copy
// when the source is dense too.  Into padded level 0: one pitched 3-D copy when the source's stream stride is a whole
// number of its rows.  Otherwise one 2-D copy per stream.
int dvfe_tracker::h2d(uint8_t* dst, size_t dst_pitch, size_t dst_stride, const uint8_t* src, size_t src_pitch, size_t src_stride,
                      size_t row) {
    const bool dense = dst_pitch == row && dst_stride == row * H;
    if (dense && src_pitch == row && src_stride == dst_stride) {
        DVFE_CUDA(cudaMemcpyAsync(dst, src, (size_t)B * dst_stride, cudaMemcpyHostToDevice, cs));
    } else if (!dense && src_stride % src_pitch == 0) {
        cudaMemcpy3DParms p;
        memset(&p, 0, sizeof(p));
        p.srcPtr = make_cudaPitchedPtr((void*)src, src_pitch, row, src_stride / src_pitch);
        p.dstPtr = make_cudaPitchedPtr((void*)dst, dst_pitch, row, dst_stride / dst_pitch);
        p.extent = make_cudaExtent(row, (size_t)H, (size_t)B);
        p.kind = cudaMemcpyHostToDevice;
        DVFE_CUDA(cudaMemcpy3DAsync(&p, cs));
    } else {
        for (int s = 0; s < B; s++)
            DVFE_CUDA(cudaMemcpy2DAsync(dst + s * dst_stride, dst_pitch, src + s * src_stride, src_pitch, row, (size_t)H,
                                        cudaMemcpyHostToDevice, cs));
    }
    return DVFE_OK;
}

StepSources slab_sources(int B, const uint8_t* left, const uint8_t* right, const uint8_t* mask, size_t stride, int pitch,
                         size_t mask_stride, int mask_pitch) {
    StepSources src;
    const uint8_t* base[3] = {left, right, mask};
    const size_t st[3] = {stride, stride, mask_stride};
    const int pt[3] = {pitch, pitch, mask_pitch};
    for (int c = 0; c < 3; c++) {
        src.img[c].assign(B, ImgSrc{nullptr, pt[c]});
        if (!base[c]) continue;
        for (int s = 0; s < B; s++) src.img[c][s].ptr = base[c] + s * st[c];
        src.uniform[c] = true;
        src.stride[c] = st[c];
    }
    return src;
}

StepSources dvfe_tracker::slab(const uint8_t* left, const uint8_t* right, const uint8_t* mask, size_t stride, int pitch) const {
    const int div = prep_active() ? in_ch : 1;
    return slab_sources(B, left, right, mask, stride, pitch, stride / (size_t)div, pitch / div);
}

int dvfe_tracker::upload_sources(const StepSources& src) {
    if (src_step == frames) return DVFE_OK;
    // h_src[par] was last the source of step k-2's copy, which has completed (wait_slot)
    ImgSrc* h = h_src[frames % 2];
    for (int c = 0; c < 3; c++) memcpy(h + (size_t)c * B, src.img[c].data(), B * sizeof(ImgSrc));
    DVFE_CUDA(cudaMemcpyAsync(d_src, h, (size_t)3 * B * sizeof(ImgSrc), cudaMemcpyHostToDevice, st));
    src_step = frames;
    return DVFE_OK;
}

// The route depends on where the images are, whether they need the ingest kernel (BGR or undistortion maps) and the width:
//   device, gray            the step copies the caller's images into level 0 itself;
//   device, ingest          the ingest kernel writes level 0 on the compute stream;
//   host, ingest            dense staging, then the ingest kernel on the upload stream;
//   host, gray, staged      dense staging, which the step copies into level 0 (pitched DMA of rows that are not a multiple
//                           of 64 bytes is slow);
//   host, gray, in place    pitched DMA straight into level 0.
// A table that is not uniform (place_table) takes the same routes image by image.
// Host routes end with ev_up[par] on the upload stream, which the compute stream waits for.  The slots written here were
// last read by step k-2, which wait_slot() has completed.
int dvfe_tracker::place_input(const StepSources& src, bool device, StepInput* in) {
    DVFE_CHECK(wait_slot());
    const bool has_right = src.any(1);
    if (!src.uniform[0] || (has_right && (!src.uniform[1] || src.stride[1] != src.stride[0] ||
                                          src.img[1][0].pitch != src.img[0][0].pitch)))
        return place_table(src, device, in);
    const uint8_t* left = src.img[0][0].ptr;
    const uint8_t* right = has_right ? src.img[1][0].ptr : nullptr;
    const size_t stream_stride = src.stride[0];
    const int pitch = src.img[0][0].pitch;
    const bool prep = prep_active();
    *in = StepInput();
    in->has_right = right != nullptr;
    if (device && !prep) {
        in->left = left; in->right = right; in->stride = stream_stride; in->pitch = pitch;
        return DVFE_OK;
    }
    const uint8_t* srcs[2] = {left, right};
    in->in_place = true;
    if (device) {
        for (int cam = 0; cam < 2; cam++)
            if (srcs[cam]) DVFE_CHECK(ingest(srcs[cam], stream_stride, pitch, cam, st));
        return DVFE_OK;
    }
    const int par = (int)(frames % 2);
    const size_t row = (size_t)W * in_ch, img = row * H;
    for (int cam = 0; cam < 2; cam++) {
        if (!srcs[cam]) continue;
        if (prep || staged_upload) {
            uint8_t* dst = d_stage[par] + (size_t)cam * B * img;
            DVFE_CHECK(h2d(dst, row, img, srcs[cam], (size_t)pitch, stream_stride, row));
            if (prep) DVFE_CHECK(ingest(dst, img, (int)row, cam, cs));
        } else {
            DVFE_CHECK(h2d(level0(cam), desc.lv[0].pitch, desc.bytes, srcs[cam], (size_t)pitch, stream_stride, row));
        }
    }
    DVFE_CUDA(cudaEventRecord(ev_up[par], cs));
    DVFE_CUDA(cudaStreamWaitEvent(st, ev_up[par], 0));
    if (!prep && staged_upload) {
        in->left = d_stage[par]; in->right = right ? d_stage[par] + B * img : nullptr;
        in->stride = img; in->pitch = W; in->in_place = false;
    }
    return DVFE_OK;
}

// Every image from where it lives, absent ones not at all.  Host: one 2-D copy per present image, into level 0 or the staging
// buffer, which the routes above then treat as a slab.  Device: the table goes to the device and the gather form of the level-0
// copy (with the border) or of the ingest kernel reads each image through it, on the compute stream.
int dvfe_tracker::place_table(const StepSources& src, bool device, StepInput* in) {
    const bool prep = prep_active();
    *in = StepInput();
    in->has_right = src.any(1);
    in->in_place = true;
    if (device) {
        DVFE_CHECK(upload_sources(src));
        for (int cam = 0; cam < 2; cam++) {
            if (!src.any(cam)) continue;
            if (prep) {
                IngestArgs a;
                a.src = nullptr; a.src_stride = 0; a.src_pitch = 0; a.ch = in_ch;
                a.map1 = maps_uniform[cam] ? stream_map1(cam, 0) : nullptr;
                a.map2 = maps_uniform[cam] ? stream_map2(cam, 0) : nullptr;
                a.dst = level0(cam);
                a.dst_stride = desc.bytes; a.dst_pitch = desc.lv[0].pitch;
                a.w = W; a.h = H; a.n_img = B; a.keep_channels = 0;
                DVFE_CHECK(launch_ingest_table(a, d_src + (size_t)cam * B, st, maps_uniform[cam] ? nullptr : d_imaps[cam]));
            } else {
                DVFE_CHECK(launch_pyr_level0_table(d_src + (size_t)cam * B, cam ? right_slot(frames) : left_slot(frames), desc.bytes,
                                                   B, desc, st));
            }
        }
        in->l0_border = !prep && pyr_level0_writes_border(desc);
        return DVFE_OK;
    }
    const int par = (int)(frames % 2);
    const size_t row = (size_t)W * in_ch, img = row * H;
    for (int cam = 0; cam < 2; cam++) {
        if (!src.any(cam)) continue;
        uint8_t* stage = d_stage[par] + (size_t)cam * B * img;
        for (int s = 0; s < B; s++) {
            const ImgSrc& e = src.img[cam][s];
            if (!e.ptr) continue;
            if (prep || staged_upload)
                DVFE_CUDA(cudaMemcpy2DAsync(stage + s * img, row, e.ptr, (size_t)e.pitch, row, (size_t)H, cudaMemcpyHostToDevice, cs));
            else
                DVFE_CUDA(cudaMemcpy2DAsync(level0(cam) + s * (size_t)desc.bytes, (size_t)desc.lv[0].pitch, e.ptr, (size_t)e.pitch, row,
                                            (size_t)H, cudaMemcpyHostToDevice, cs));
        }
        if (prep) DVFE_CHECK(ingest(stage, img, (int)row, cam, cs));
    }
    DVFE_CUDA(cudaEventRecord(ev_up[par], cs));
    DVFE_CUDA(cudaStreamWaitEvent(st, ev_up[par], 0));
    if (!prep && staged_upload) {
        in->left = d_stage[par]; in->right = in->has_right ? d_stage[par] + B * img : nullptr;
        in->stride = img; in->pitch = W; in->in_place = false;
    }
    return DVFE_OK;
}

// the staging buffers the host routes of the current input format need: [2 cameras][B][H*W*in_ch] when images are staged or
// ingested, none when they are DMA'd into level 0
int dvfe_tracker::size_stage() {
    for (int p = 0; p < 2; p++) { cudaFree(d_stage[p]); d_stage[p] = nullptr; }
    if (!staged_upload && !prep_active()) return DVFE_OK;
    for (int p = 0; p < 2; p++) DVFE_CUDA(cudaMalloc((void**)&d_stage[p], (size_t)2 * B * W * H * in_ch));
    return DVFE_OK;
}

int grp_set_input(dvfe_tracker* t, int channels);
int grp_set_maps(dvfe_tracker* t, int cam, const int16_t* map1, const uint16_t* map2);
int grp_set_stream_camera(dvfe_tracker* t, int stream, const dvfe_camera* cam0, const dvfe_camera* cam1);
int grp_set_stream_maps(dvfe_tracker* t, int stream, int cam, const int16_t* map1, const uint16_t* map2);

extern "C" int dvfe_set_input(dvfe_tracker* t, int channels) {
    if (!t || (channels != 1 && channels != 3)) { dvfe_set_error("set_input: channels must be 1 (gray) or 3 (BGR)"); return DVFE_ERR_INVALID; }
    if (IS_GROUP(t)) return grp_set_input(t, channels);
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    DVFE_CHECK(t->wait_all());
    DVFE_CUDA(cudaStreamSynchronize(t->cs));
    t->in_ch = channels;
    return t->size_stage();
}

extern "C" int dvfe_set_undistort_maps(dvfe_tracker* t, int cam, const int16_t* map1, const uint16_t* map2) {
    if (!t || cam < 0 || cam > 1 || (map1 != nullptr) != (map2 != nullptr)) { dvfe_set_error("set_undistort_maps: bad argument"); return DVFE_ERR_INVALID; }
    if (IS_GROUP(t)) return grp_set_maps(t, cam, map1, map2);
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    DVFE_CHECK(t->wait_all());
    DVFE_CUDA(cudaStreamSynchronize(t->cs));
    cudaFree(t->d_map1[cam]); cudaFree(t->d_map2[cam]);
    t->d_map1[cam] = nullptr; t->d_map2[cam] = nullptr;
    if (map1) {
        const size_t P = (size_t)t->W * t->H;
        DVFE_CUDA(cudaMalloc((void**)&t->d_map1[cam], P * 4));
        DVFE_CUDA(cudaMalloc((void**)&t->d_map2[cam], P * 2));
        DVFE_CUDA(cudaMemcpy(t->d_map1[cam], map1, P * 4, cudaMemcpyHostToDevice));
        DVFE_CUDA(cudaMemcpy(t->d_map2[cam], map2, P * 2, cudaMemcpyHostToDevice));
    }
    for (int s = 0; s < t->B; s++) {                 // every stream follows the shared maps again
        cudaFree(t->s_map1[cam][s]); cudaFree(t->s_map2[cam][s]);
        t->s_map1[cam][s] = nullptr; t->s_map2[cam][s] = nullptr;
        t->own_maps[cam][s] = 0;
    }
    DVFE_CHECK(t->update_maps(cam));
    return t->size_stage();
}

// Per-stream maps live in device memory the call allocates, so no step may be in flight; the call does not wait for one itself,
// which would take the records of the earlier steps from the caller's later dvfe_wait calls.
extern "C" int dvfe_set_stream_undistort_maps(dvfe_tracker* t, int stream, int cam, const int16_t* map1, const uint16_t* map2) {
    if (!t || cam < 0 || cam > 1 || (map1 != nullptr) != (map2 != nullptr)) {
        dvfe_set_error("set_stream_undistort_maps: bad argument");
        return DVFE_ERR_INVALID;
    }
    if (IS_GROUP(t)) return grp_set_stream_maps(t, stream, cam, map1, map2);
    if (stream < 0 || stream >= t->B) { dvfe_set_error("set_stream_undistort_maps: bad stream index %d", stream); return DVFE_ERR_INVALID; }
    if (t->completed < t->frames) {
        dvfe_set_error("set_stream_undistort_maps: %ld step(s) in flight; wait for them first", t->frames - t->completed);
        return DVFE_ERR_INVALID;
    }
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    DVFE_CUDA(cudaStreamSynchronize(t->st));
    DVFE_CUDA(cudaStreamSynchronize(t->cs));
    short* m1 = nullptr;
    unsigned short* m2 = nullptr;
    if (map1) {
        const size_t P = (size_t)t->W * t->H;
        cudaError_t e = cudaMalloc((void**)&m1, P * 4);
        if (e == cudaSuccess) e = cudaMalloc((void**)&m2, P * 2);
        if (e == cudaSuccess) e = cudaMemcpy(m1, map1, P * 4, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(m2, map2, P * 2, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            cudaFree(m1); cudaFree(m2);
            dvfe_set_error("set_stream_undistort_maps: %s", cudaGetErrorString(e));
            return DVFE_ERR_CUDA;
        }
    }
    cudaFree(t->s_map1[cam][stream]); cudaFree(t->s_map2[cam][stream]);
    t->s_map1[cam][stream] = m1; t->s_map2[cam][stream] = m2;
    t->own_maps[cam][stream] = 1;
    DVFE_CHECK(t->update_maps(cam));
    return t->size_stage();
}

static bool camera_ok(const dvfe_camera* c) {
    const double v[8] = {c->fx, c->fy, c->cx, c->cy, c->k1, c->k2, c->p1, c->p2};
    for (double x : v)
        if (!isfinite(x)) return false;
    return c->fx != 0.0 && c->fy != 0.0;
}

// The calibration of the next step submitted; steps already submitted keep theirs (submit() uploads the table).  No tracking state
// is touched.
extern "C" int dvfe_set_stream_camera(dvfe_tracker* t, int stream, const dvfe_camera* cam0, const dvfe_camera* cam1) {
    if (!t || !cam0) { dvfe_set_error("set_stream_camera: null argument"); return DVFE_ERR_INVALID; }
    if (!camera_ok(cam0) || (cam1 && !camera_ok(cam1))) {
        dvfe_set_error("set_stream_camera: camera parameters must be finite, with fx and fy non-zero");
        return DVFE_ERR_INVALID;
    }
    if (IS_GROUP(t)) return grp_set_stream_camera(t, stream, cam0, cam1);
    if (stream < 0 || stream >= t->B) { dvfe_set_error("set_stream_camera: bad stream index %d", stream); return DVFE_ERR_INVALID; }
    t->cams[stream] = make_cam(*cam0);
    t->cams[(size_t)t->B + stream] = make_cam(cam1 ? *cam1 : *cam0);
    t->cam_dirty = true;
    return DVFE_OK;
}

static int check_step_args(dvfe_tracker* t, const uint8_t* left, int pitch, const double* time0) {
    const int in_ch = !t ? 1 : (t->groups.empty() ? t->in_ch : t->groups[0]->in_ch);
    if (!t || !left || !time0 || pitch < t->W * in_ch) {
        dvfe_set_error("track: input wrong, received at least one empty parameter");   // feature_utils.cpp:39-41
        return DVFE_ERR_INVALID;
    }
    return DVFE_OK;
}

// one raw step of a leaf tracker, enqueued; sflags: per-stream DVFE_FRAME_* (validated) or null
int leaf_track(dvfe_tracker* t, const StepSources& src, const double* time0, const uint8_t* sflags, bool device) {
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    t->src_step = -1;                       // this step's table is not on the device yet
    StepInput in;
    DVFE_CHECK(t->place_input(src, device, &in));
    return t->submit(in, time0, false, sflags);
}

static int wait_all_steps(dvfe_tracker* t) {
    if (IS_GROUP(t)) return grp_wait_all(t);
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    return t->wait_all();
}

extern "C" int dvfe_track_image_async(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, size_t stream_stride,
                                      int pitch, const double* time0) {
    return dvfe_track_image_ex(t, left, right, stream_stride, pitch, time0, nullptr, 0u);
}

extern "C" int dvfe_wait(dvfe_tracker* t) {
    if (!t) { dvfe_set_error("wait: null tracker"); return DVFE_ERR_INVALID; }
    if (IS_GROUP(t)) return grp_wait(t);
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    return t->wait_one();
}

extern "C" int dvfe_track_image(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, size_t stream_stride,
                                int pitch, const double* time0) {
    DVFE_CHECK(dvfe_track_image_ex(t, left, right, stream_stride, pitch, time0, nullptr, 0u));
    return wait_all_steps(t);
}

extern "C" int dvfe_track_image_device(dvfe_tracker* t, const uint8_t* d_left, const uint8_t* d_right,
                                       size_t stream_stride, int pitch, const double* time0) {
    DVFE_CHECK(check_step_args(t, d_left, pitch, time0));
    // an earlier step's capacity error is reported here, before this step is enqueued
    DVFE_CHECK(wait_all_steps(t));
    DVFE_CHECK(dvfe_track_image_ex(t, d_left, d_right, stream_stride, pitch, time0, nullptr, DVFE_STEP_DEVICE_INPUT));
    return wait_all_steps(t);
}

extern "C" int dvfe_track_image_device_async(dvfe_tracker* t, const uint8_t* d_left, const uint8_t* d_right,
                                             size_t stream_stride, int pitch, const double* time0) {
    return dvfe_track_image_ex(t, d_left, d_right, stream_stride, pitch, time0, nullptr, DVFE_STEP_DEVICE_INPUT);
}

int check_stream_flags(const uint8_t* stream_flags, int B, const char* who, const uint8_t** out) {
    bool any = false;
    if (stream_flags)
        for (int s = 0; s < B; s++) {
            const unsigned f = stream_flags[s];
            if ((f & ~(DVFE_FRAME_SKIP | DVFE_FRAME_NO_RIGHT | DVFE_FRAME_RESET)) ||
                (f & (DVFE_FRAME_SKIP | DVFE_FRAME_RESET)) == (DVFE_FRAME_SKIP | DVFE_FRAME_RESET)) {
                dvfe_set_error("%s: stream %d: invalid stream flags 0x%x", who, s, f);
                return DVFE_ERR_INVALID;
            }
            any = any || f != 0;
        }
    *out = any ? stream_flags : nullptr;                       // no flag set: exactly the step of the plain entry points
    return DVFE_OK;
}

extern "C" int dvfe_track_image_ex(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, size_t stream_stride, int pitch,
                                   const double* time0, const uint8_t* stream_flags, unsigned flags) {
    DVFE_CHECK(check_step_args(t, left, pitch, time0));
    if (flags & ~DVFE_STEP_DEVICE_INPUT) { dvfe_set_error("track_image_ex: unknown flags 0x%x", flags); return DVFE_ERR_INVALID; }
    const bool device = (flags & DVFE_STEP_DEVICE_INPUT) != 0;
    const uint8_t* sf = nullptr;
    DVFE_CHECK(check_stream_flags(stream_flags, t->B, "track_image_ex", &sf));
    if (IS_GROUP(t)) return grp_track_image_ex(t, left, right, stream_stride, pitch, time0, sf, device);
    return leaf_track(t, t->slab(left, right, nullptr, stream_stride, pitch), time0, sf, device);
}

extern "C" int dvfe_set_lk_mode_site(dvfe_tracker* t, int site, int back_max_level, double fb_threshold) {
    if (!t || site < -1 || site > DVFE_LK_SEMANTIC_STEREO || back_max_level < 0 || back_max_level >= DVFE_MAX_PYR_LEVELS ||
        !(fb_threshold > 0.0)) {
        dvfe_set_error("set_lk_mode: bad argument");
        return DVFE_ERR_INVALID;
    }
    if (IS_GROUP(t)) return grp_set_lk_mode(t, site, back_max_level, fb_threshold);
    for (int i = 0; i < 4; i++)
        if (site < 0 || site == i) { t->lk_back_level[i] = back_max_level; t->lk_fb_thresh[i] = fb_threshold; }
    t->drop_graphs();                 // the captured steps carry the old parameters
    return DVFE_OK;
}

extern "C" int dvfe_set_lk_mode(dvfe_tracker* t, int back_max_level, double fb_threshold) {
    return dvfe_set_lk_mode_site(t, -1, back_max_level, fb_threshold);
}

extern "C" int dvfe_set_detect_mode(dvfe_tracker* t, int mode) {
    if (!t || (mode != DVFE_DETECT_CPU && mode != DVFE_DETECT_CUDA)) { dvfe_set_error("set_detect_mode: bad argument"); return DVFE_ERR_INVALID; }
    if (IS_GROUP(t)) return grp_set_detect_mode(t, mode);
    t->detect_cuda = mode == DVFE_DETECT_CUDA;
    t->drop_graphs();                 // the captured steps carry the old job table
    return DVFE_OK;
}

extern "C" int dvfe_set_reject_with_f(dvfe_tracker* t, double f_threshold) {
    if (!t || !isfinite(f_threshold) || f_threshold < 0.0) {
        dvfe_set_error("set_reject_with_f: the threshold must be finite and >= 0 (0 = off)");
        return DVFE_ERR_INVALID;
    }
    if (IS_GROUP(t)) return grp_set_reject_with_f(t, f_threshold);
    if (f_threshold == t->reject_f) return DVFE_OK;
    if (f_threshold > 0.0 && !t->d_fm_models) {       // steps in flight never read it: they were enqueued with the mode off
        DVFE_CUDA(cudaSetDevice(t->cfg.device));
        DVFE_CUDA(cudaMalloc((void**)&t->d_fm_models, reject_with_f_models(t->B) * sizeof(double)));
    }
    t->reject_f = f_threshold;
    t->drop_graphs();                 // the captured steps carry the old threshold (or no rejection)
    return DVFE_OK;
}

int dvfe_tracker::semantic_submit(const StepSources& src, const int* exist_inst, const double* time0, unsigned flags,
                                  const uint8_t* sflags) {
    DVFE_CHECK(wait_slot());                // before the mask copy: d_inv_in[par] / d_labels[par] are step k-2's until then
    src_step = -1;                          // this step's table is not on the device yet
    const size_t P = (size_t)W * H;
    const int par = (int)(frames % 2);
    const bool device = (flags & DVFE_DYN_DEVICE_INPUT) != 0, labels = (flags & DVFE_DYN_LABELS) != 0;
    const std::vector<ImgSrc>& mask = src.img[2];
    // a skipped stream counts as one without instances: its mask is neither copied nor eroded
    bool all = true;
    for (int s = 0; s < B; s++) {
        const bool ex = !(sflags && (sflags[s] & DVFE_FRAME_SKIP)) && exist_inst[s];
        h_exist[par][s] = ex ? 1 : 0;
        all = all && ex;
        if (ex && !mask[s].ptr) { dvfe_set_error("track_semantic_image: exist_inst set but no mask"); return DVFE_ERR_INVALID; }
    }
    // where the erosion reads the mask / label image from
    const uint8_t* d_mask = src.uniform[2] ? mask[0].ptr : nullptr;
    size_t d_mask_stride = src.stride[2];
    int d_mask_pitch = mask[0].pitch;
    if (!device || (!src.uniform[2] && src.any(2))) {
        // host: mask -> device on the upload stream, ahead of the images (one copy when every stream has one);
        // device masks that are not one slab: gathered on the compute stream
        if (labels && !d_labels[par]) DVFE_CUDA(cudaMalloc((void**)&d_labels[par], (size_t)B * P));
        uint8_t* dst = labels ? d_labels[par] : d_inv_in[par];
        if (device) {
            DVFE_CHECK(upload_sources(src));
            DVFE_CHECK(launch_gather_images(d_src + (size_t)2 * B, dst, P, W, W, H, B, st));
        } else if (all && src.uniform[2] && mask[0].pitch == W && src.stride[2] == P) {
            DVFE_CUDA(cudaMemcpyAsync(dst, mask[0].ptr, (size_t)B * P, cudaMemcpyHostToDevice, cs));
        } else {
            for (int s = 0; s < B; s++)
                if (h_exist[par][s])
                    DVFE_CUDA(cudaMemcpy2DAsync(dst + s * P, W, mask[s].ptr, mask[s].pitch, W, (size_t)H, cudaMemcpyHostToDevice, cs));
        }
        d_mask = dst; d_mask_stride = P; d_mask_pitch = W;
    }
    StepInput in;                           // a host route's ev_up, recorded after the images, covers the mask copy too
    DVFE_CHECK(place_input(src, device, &in));
    lab_ptr[par] = labels ? d_mask : nullptr; lab_stride[par] = d_mask_stride; lab_pitch[par] = d_mask_pitch;
    DVFE_CUDA(cudaMemcpyAsync(d_exist, h_exist[par], B * sizeof(int), cudaMemcpyHostToDevice, st));
    // region mask = exist_inst ? erode(inv_merge_mask, mask_morphology_size) : all 255   (:764-772); with a label image
    // inv_merge_mask = (no instance bit set ? 255 : 0) is formed while it is read (basic/semantic_image.cpp:31-38)
    const int k = cfg.use_mask_morphology ? cfg.mask_morphology_size : 1;
    if (d_mask != nullptr)
        DVFE_CHECK(launch_erode_rect(d_mask, d_mask_pitch, d_region, W, d_region_tmp, W, H, k < 1 ? 1 : k, B, d_mask_stride, d_exist,
                                     st, labels ? 1 : 0));
    else
        DVFE_CHECK(launch_erode_rect(d_inv_in[par], W, d_region, W, d_region_tmp, W, H, 1, B, P, d_exist, st));   // all 255
    if (sflags && inst)
        for (int s = 0; s < B; s++)
            if (sflags[s] & DVFE_FRAME_RESET) reset_instances(s);
    return submit(in, time0, true, sflags);
}

extern "C" int dvfe_track_semantic_ex(dvfe_tracker* t, const uint8_t* left, const uint8_t* right, const uint8_t* inv_merge_mask,
                                      size_t stream_stride, int pitch, const int* exist_inst, const double* time0,
                                      const uint8_t* stream_flags, unsigned flags) {
    DVFE_CHECK(check_step_args(t, left, pitch, time0));
    if (!exist_inst) { dvfe_set_error("track_semantic_image: exist_inst is null"); return DVFE_ERR_INVALID; }
    if (flags & ~DVFE_DYN_DEVICE_INPUT) { dvfe_set_error("track_semantic_ex: unknown flags 0x%x", flags); return DVFE_ERR_INVALID; }
    const uint8_t* sf = nullptr;
    DVFE_CHECK(check_stream_flags(stream_flags, t->B, "track_semantic_ex", &sf));
    if (IS_GROUP(t)) return grp_track_semantic(t, left, right, inv_merge_mask, stream_stride, pitch, exist_inst, time0, sf, flags);
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    return t->semantic_submit(t->slab(left, right, inv_merge_mask, stream_stride, pitch), exist_inst, time0, flags, sf);
}

extern "C" int dvfe_track_semantic_image(dvfe_tracker* t, const uint8_t* left, const uint8_t* right,
                                         const uint8_t* inv_merge_mask, size_t stream_stride, int pitch,
                                         const int* exist_inst, const double* time0) {
    DVFE_CHECK(check_step_args(t, left, pitch, time0));
    DVFE_CHECK(wait_all_steps(t));
    DVFE_CHECK(dvfe_track_semantic_ex(t, left, right, inv_merge_mask, stream_stride, pitch, exist_inst, time0, nullptr, 0u));
    return wait_all_steps(t);
}

extern "C" int dvfe_get_features(dvfe_tracker* t, int stream, dvfe_obs* out, int cap, int* n_out) {
    if (IS_GROUP(t)) {
        dvfe_tracker* leaf; int local;
        DVFE_CHECK(grp_route(t, stream, &leaf, &local));
        return dvfe_get_features(leaf, local, out, cap, n_out);
    }
    if (!t || stream < 0 || stream >= t->B || !n_out) { dvfe_set_error("get_features: bad argument"); return DVFE_ERR_INVALID; }
    const int n = t->h_nobs[t->out_slot][stream];
    *n_out = n;
    if (n > cap) { dvfe_set_error("get_features: %d records, capacity %d", n, cap); return DVFE_ERR_CAPACITY; }
    if (n > 0 && out) memcpy(out, t->h_obs[t->out_slot] + (size_t)stream * 2 * t->cap, (size_t)n * sizeof(dvfe_obs));
    return DVFE_OK;
}

// ---- state get/set (teacher-forced parity tests, checkpointing) ---------------------------------------
extern "C" int dvfe_get_state(dvfe_tracker* t, int stream, dvfe_state* stt, int cap) {
    if (IS_GROUP(t)) {
        dvfe_tracker* leaf; int local;
        DVFE_CHECK(grp_route(t, stream, &leaf, &local));
        return dvfe_get_state(leaf, local, stt, cap);
    }
    if (!t || !stt || stream < 0 || stream >= t->B) { dvfe_set_error("get_state: bad argument"); return DVFE_ERR_INVALID; }
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    DVFE_CHECK(t->wait_all());
    DVFE_CUDA(cudaStreamSynchronize(t->st));
    int n = 0;
    DVFE_CUDA(cudaMemcpy(&n, t->bg.n + stream, sizeof(int), cudaMemcpyDeviceToHost));
    DVFE_CUDA(cudaMemcpy(&stt->next_id, t->d_next_id + stream, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    stt->n = n;
    stt->prev_time = t->prev_time[stream];
    if (n > cap) { dvfe_set_error("get_state: %d points, capacity %d", n, cap); return DVFE_ERR_CAPACITY; }
    const size_t o = (size_t)stream * t->cap;
    if (n > 0) {
        if (stt->ids) DVFE_CUDA(cudaMemcpy(stt->ids, t->bg.ids + o, n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        if (stt->track_cnt) DVFE_CUDA(cudaMemcpy(stt->track_cnt, t->bg.track_cnt + o, n * sizeof(int32_t), cudaMemcpyDeviceToHost));
        if (stt->last_points) DVFE_CUDA(cudaMemcpy(stt->last_points, t->bg.pts + o, n * sizeof(float2), cudaMemcpyDeviceToHost));
        if (stt->prev_un) DVFE_CUDA(cudaMemcpy(stt->prev_un, t->bg.un + o, n * sizeof(float2), cudaMemcpyDeviceToHost));
        if (stt->right_prev_un) DVFE_CUDA(cudaMemcpy(stt->right_prev_un, t->bg.rprev_un + o, n * sizeof(float2), cudaMemcpyDeviceToHost));
        if (stt->right_prev_valid) DVFE_CUDA(cudaMemcpy(stt->right_prev_valid, t->bg.rprev_valid + o, n, cudaMemcpyDeviceToHost));
    }
    return DVFE_OK;
}

extern "C" int dvfe_set_state(dvfe_tracker* t, int stream, const dvfe_state* stt) {
    if (IS_GROUP(t)) {
        dvfe_tracker* leaf; int local;
        DVFE_CHECK(grp_route(t, stream, &leaf, &local));
        return dvfe_set_state(leaf, local, stt);
    }
    if (!t || !stt || stream < 0 || stream >= t->B || stt->n < 0 || stt->n > t->cap) {
        dvfe_set_error("set_state: bad argument");
        return DVFE_ERR_INVALID;
    }
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    DVFE_CHECK(t->wait_all());
    DVFE_CUDA(cudaStreamSynchronize(t->st));
    const int n = stt->n;
    const size_t o = (size_t)stream * t->cap;
    DVFE_CUDA(cudaMemcpy(t->bg.n + stream, &n, sizeof(int), cudaMemcpyHostToDevice));
    DVFE_CUDA(cudaMemcpy(t->d_next_id + stream, &stt->next_id, sizeof(uint32_t), cudaMemcpyHostToDevice));
    t->prev_time[stream] = stt->prev_time;
    t->tcache_valid = false;                 // the cached templates belong to the points that were just replaced
    t->tc_valid[stream] = 0;
    if (n > 0) {
        DVFE_CUDA(cudaMemcpy(t->bg.ids + o, stt->ids, n * sizeof(uint32_t), cudaMemcpyHostToDevice));
        DVFE_CUDA(cudaMemcpy(t->bg.track_cnt + o, stt->track_cnt, n * sizeof(int32_t), cudaMemcpyHostToDevice));
        DVFE_CUDA(cudaMemcpy(t->bg.pts + o, stt->last_points, n * sizeof(float2), cudaMemcpyHostToDevice));
        DVFE_CUDA(cudaMemcpy(t->bg.un + o, stt->prev_un, n * sizeof(float2), cudaMemcpyHostToDevice));
        DVFE_CUDA(cudaMemcpy(t->bg.rprev_un + o, stt->right_prev_un, n * sizeof(float2), cudaMemcpyHostToDevice));
        DVFE_CUDA(cudaMemcpy(t->bg.rprev_valid + o, stt->right_prev_valid, n, cudaMemcpyHostToDevice));
    }
    return DVFE_OK;
}

extern "C" int dvfe_set_stream(dvfe_tracker* t, void* cuda_stream) {
    if (!t) { dvfe_set_error("set_stream: null tracker"); return DVFE_ERR_INVALID; }
    if (IS_GROUP(t)) return dvfe_set_stream(t->groups[0], cuda_stream);      // the other groups keep private streams
    DVFE_CUDA(cudaSetDevice(t->cfg.device));
    DVFE_CHECK(t->wait_all());
    DVFE_CUDA(cudaStreamSynchronize(t->st));
    t->drop_graphs();
    if (t->own_stream && t->st) cudaStreamDestroy(t->st);
    t->st = (cudaStream_t)cuda_stream;
    t->own_stream = false;
    return DVFE_OK;
}

extern "C" int dvfe_profile(dvfe_tracker* t, int enable) {
    if (!t) { dvfe_set_error("profile: null tracker"); return DVFE_ERR_INVALID; }
    if (IS_GROUP(t)) return grp_profile(t, enable);
    t->prof = enable != 0;
    if (enable) {
        for (int i = 0; i < dvfe_tracker::ST_COUNT; i++) t->prof_ms[i] = 0.0;
        t->prof_steps = 0;
    }
    return DVFE_OK;
}

extern "C" int dvfe_profile_read(dvfe_tracker* t, const char** names, double* total_ms, long* steps) {
    static const char* kNames[dvfe_tracker::ST_COUNT] = {"pyramid", "lk_temporal", "compact", "gftt_mask_fill", "gftt_discs",
                                                         "gftt_response", "gftt_select", "left_post", "lk_stereo", "pack",
                                                         "d2h"};
    if (!t) { dvfe_set_error("profile_read: null tracker"); return DVFE_ERR_INVALID; }
    if (IS_GROUP(t)) return grp_profile_read(t, names, total_ms, steps);
    for (int i = 0; i < dvfe_tracker::ST_COUNT; i++) {
        if (names) names[i] = kNames[i];
        if (total_ms) total_ms[i] = t->prof_ms[i];
    }
    if (steps) *steps = t->prof_steps;
    return dvfe_tracker::ST_COUNT;
}
