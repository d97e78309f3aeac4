// Per-stream frame presence (dvfe_track_image_ex): a "partial" step, in which some streams have no frame (SKIP), no right
// image (NO_RIGHT) or start over (RESET), runs the kernels of the full step unchanged on job tables derived from the stream
// flags.  Two kernels are added to the step: the table builder at its start and the carry of the skipped streams' previous
// left pyramids after the left pyramid build.
#include "kernels.cuh"

// One thread per stream.  The tables point at the same buffers as the phase's full tables; a stream a table leaves out gets a
// point count of 0 (LK: nothing to track) or max_cnt = 0 (GFTT: gftt_job_active is false, so no kernel of the detector touches
// its mask, counters, points or ids).  What a table entry points at depends only on the flags, never on a point count, so the
// tables are built before the step changes any count.
__global__ void k_partial_tables(PartialTables p, const uint8_t* __restrict__ sflags, int n_streams, int stereo_now) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_streams) return;
    const unsigned f = sflags[s];
    const bool skip = (f & DVFE_FRAME_SKIP) != 0, reset = (f & DVFE_FRAME_RESET) != 0;
    const bool stereo = stereo_now && !skip && (f & DVFE_FRAME_NO_RIGHT) == 0;
    if (reset) {                       // a newly created tracker: no points, InstFeat::global_id_count{1}
        p.n[s] = 0;
        p.next_id[s] = 1u;
    }
    LkGroup G = p.full_temporal[s];
    if (skip) G.n = p.zero;
    // a stale forward-template cache (the stream's last present frame had no stereo step, or its points were replaced) is
    // rebuilt by k_lk_track from the image, which it does whenever the table carries no cache
    if (!(f & SF_TCACHE_VALID) || reset) G.tcache = nullptr;
    p.temporal[s] = G;
    G = p.full_stereo[s];
    if (!stereo) G.n = p.zero;
    p.stereo[s] = G;
    GfttJob J = p.full_jobs[s];
    if (skip) J.max_cnt = 0;
    p.jobs[s] = J;
    p.lane[s] = skip ? 0 : (uint8_t)(LANE_PRESENT | (stereo ? LANE_STEREO : 0));
}

int launch_partial_tables(const PartialTables& p, const uint8_t* d_sflags, int n_streams, int stereo_now, cudaStream_t st) {
    if (n_streams <= 0) return DVFE_OK;
    DVFE_LAUNCH(k_partial_tables, (n_streams + 63) / 64, 64, 0, st, p, d_sflags, n_streams, stereo_now);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

// cur[s] = prev[s] for every skipped stream s: the whole pyramid (every level with its border, `bytes` a multiple of 256), so
// the stream's next present frame tracks from its last present image while the slot rotation stays the same for all streams.
__global__ void __launch_bounds__(256) k_carry_pyramids(uint4* __restrict__ cur, const uint4* __restrict__ prev, size_t n16,
                                                        const uint8_t* __restrict__ sflags) {
    const int s = blockIdx.y;
    if (!(sflags[s] & DVFE_FRAME_SKIP)) return;
    const size_t o = (size_t)s * n16;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x)
        cur[o + i] = prev[o + i];
}

int launch_carry_pyramids(uint8_t* cur, const uint8_t* prev, size_t bytes, const uint8_t* d_sflags, int n_streams, cudaStream_t st) {
    if (n_streams <= 0) return DVFE_OK;
    const size_t n16 = bytes / 16;
    int bx = (int)((n16 + 256 * 8 - 1) / (256 * 8));
    if (bx > 128) bx = 128;
    DVFE_LAUNCH(k_carry_pyramids, dim3(bx, n_streams), 256, 0, st, (uint4*)cur, (const uint4*)prev, n16, d_sflags);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}
