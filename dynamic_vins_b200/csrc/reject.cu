// Epipolar outlier rejection inside the frame step (dvfe_set_reject_with_f): VINS-Mono's rejectWithF, i.e.
// FeatureTracker::RejectWithF (dynamic_vins/src/front_end/background_tracker.cpp:520-550, commented out there), for every stream
// of the step, between the temporal LK and the compaction (ReduceVector).
//
// One CTA per stream.  The survivors of the temporal LK (status != 0, in order) are lifted with the stream's cam0, re-projected
// with the virtual focal length 460 about the image centre and kept in shared memory; then the sequential loop of
// cv::findFundamentalMat(cur, prev, FM_RANSAC, threshold, 0.99) runs as in the seam op (geometry.cu, k_reject_with_f), whose
// comment explains why it splits into chunks of candidate samples.  Two things differ, both for the step's critical path:
//   - the first chunk holds RF_FIRST_CHUNK samples and each later one four times as many, up to RF_THREADS: with few outliers the
//     adaptive iteration budget stops within a handful of samples (after the first one when every point fits), so thread 0 does
//     not replay the RNG for 256 samples first and the warps do not score samples the loop never reaches;
//   - RANSAC scores each root warp-parallel over the points (the seam op counts with one thread per sample).
// Neither changes a result: the samples drawn depend only on the RNG and the points, inlier counts are integers, the per-point
// error is the same fm_error, and the bookkeeping runs in sample order on one thread.  The rejected survivors get status 0, so the
// compaction that follows removes them exactly as it removes LK failures (its old-index map stays right).
#include "fm.cuh"
#include "state.cuh"

#define RF_THREADS 256           // threads per CTA = candidate samples of a full chunk
#define RF_FIRST_CHUNK 8         // candidate samples of the first chunk (one per warp)

namespace {

// S.status of set s is cleared for its rejected survivors.  lanes (nullable): 0 = the stream was skipped (its status bytes are
// stale and are not read).  models: RF_THREADS * 27 doubles per set, the roots of the current chunk.
__global__ void __launch_bounds__(RF_THREADS, 1) k_reject_with_f_step(PointSetArrays S, int cap,
                                                                      const CamParams* __restrict__ cams,
                                                                      const uint8_t* __restrict__ lanes, double half_col,
                                                                      double half_row, double threshold, double* models_all) {
    extern __shared__ float2 s_pts[];                       // [cap] current, [cap] previous, then [cap] source indices
    __shared__ unsigned short s_idx[RF_THREADS][FM_MODEL_POINTS];
    __shared__ signed char s_nmodels[RF_THREADS];           // -1: sample rejected (collinear), else number of roots
    __shared__ float s_score[RF_THREADS][3];                // RANSAC: inlier count; LMedS: median error
    __shared__ int s_warp[RF_THREADS / 32];
    __shared__ int s_m, s_done, s_found, s_best_slot, s_best_root;
    __shared__ double s_best[9], s_min_median;
    const int set = blockIdx.x;
    if (lanes != nullptr && !lanes[set]) return;
    const int n = S.n[set];
    if (n < 8) return;                                      // fewer than 8 survivors: no rejection (VINS-Mono's guard)
    const size_t o = (size_t)set * cap;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float2* m1 = s_pts;                                     // findFundamentalMat's points1: current positions
    float2* m2 = s_pts + cap;                               // points2: previous positions
    unsigned short* src = reinterpret_cast<unsigned short*>(s_pts + 2 * cap);
    const CamParams cam = cams[set];

    // the survivors in order (ReduceVector's order), re-projected
    if (tid == 0) s_m = 0;
    __syncthreads();
    for (int c0 = 0; c0 < n; c0 += RF_THREADS) {
        const int i = c0 + tid;
        const bool keep = i < n && S.status[o + i] != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        int off = s_m;
        for (int w = 0; w < warp; w++) off += s_warp[w];
        if (keep) {
            const int j = off + __popc(bal & ((1u << lane) - 1u));
            m1[j] = fm_reproject(cam, S.lk_out[o + i], half_col, half_row);
            m2[j] = fm_reproject(cam, S.pts[o + i], half_col, half_row);
            src[j] = (unsigned short)i;
        }
        __syncthreads();
        if (tid == 0) {
            int t = 0;
            for (int w = 0; w < RF_THREADS / 32; w++) t += s_warp[w];
            s_m += t;
        }
        __syncthreads();
    }
    const int m = s_m;
    if (m < 8) return;
    const bool lmeds = m < 15;
    const float t_ransac = (float)(threshold * threshold);
    double* models = models_all + (size_t)set * RF_THREADS * 27;

    // thread 0 carries the sequential state of the OpenCV loop
    FmRng rng{~0ull};
    int niters = FM_MAX_ITERS, iter = 0, max_good = 0, failed_attempts = 0;
    bool found = false;
    if (tid == 0) {
        s_done = 0; s_min_median = 1.7976931348623157e308;
        if (lmeds) { niters = fm_update_iters(0.99, 0.45, FM_MODEL_POINTS, FM_MAX_ITERS); if (niters < 3) niters = 3; }
    }
    const int max_attempts = lmeds ? 1000 : 10000;         // getSubset's give-up bound per iteration
    int chunk = RF_FIRST_CHUNK;
    for (;;) {
        // (a) the RNG stream: `chunk` candidate samples, duplicates inside a sample redrawn
        if (tid == 0) {
            for (int a = 0; a < chunk; a++)
                for (int i = 0; i < FM_MODEL_POINTS; i++) {
                    int v;
                    bool dup;
                    do {
                        v = rng.uniform(0, m);
                        dup = false;
                        for (int j = 0; j < i; j++) dup |= s_idx[a][j] == v;
                    } while (dup);
                    s_idx[a][i] = (unsigned short)v;
                }
        }
        __syncthreads();
        // (b) one candidate sample per thread: collinearity test and 7-point solve (LMedS: the medians too, n <= 14)
        if (tid < chunk) {
            int idx[FM_MODEL_POINTS];
            for (int i = 0; i < FM_MODEL_POINTS; i++) idx[i] = s_idx[tid][i];
            int k = -1;
            if (!fm_collinear(m1, idx) && !fm_collinear(m2, idx)) {
                double F[27];
                k = fm_run7(m1, m2, idx, F);
                for (int r = 0; r < k; r++) {
                    const double* Fr = F + 9 * r;
                    if (lmeds) {
                        float e[14];
                        for (int j = 0; j < m; j++) {                 // insertion sort, m <= 14
                            const float v = fm_error(Fr, m1[j], m2[j]);
                            int q = j;
                            while (q > 0 && e[q - 1] > v) { e[q] = e[q - 1]; q--; }
                            e[q] = v;
                        }
                        s_score[tid][r] = e[m / 2];                   // std::nth_element(..., count / 2)
                    }
                    for (int q = 0; q < 9; q++) models[27 * tid + 9 * r + q] = Fr[q];
                }
            }
            s_nmodels[tid] = (signed char)k;
        }
        __syncthreads();
        // (c) RANSAC: the inliers of every root, one warp per sample, lanes over the points
        if (!lmeds) {
            for (int a = warp; a < chunk; a += RF_THREADS / 32) {
                const int k = s_nmodels[a];
                for (int r = 0; r < k; r++) {
                    double F[9];
                    for (int q = 0; q < 9; q++) F[q] = models[27 * a + 9 * r + q];
                    int good = 0;
                    for (int j = lane; j < m; j += 32) good += fm_error(F, m1[j], m2[j]) <= t_ransac;
                    good = __reduce_add_sync(0xffffffffu, good);
                    if (lane == 0) s_score[a][r] = (float)good;
                }
            }
            __syncthreads();
        }
        // (d) OpenCV's loop bookkeeping replayed over the chunk in sample order
        if (tid == 0) {
            int best_slot = -1, best_root = 0;
            for (int a = 0; a < chunk && !s_done; a++) {
                if (iter >= niters) { s_done = 1; break; }
                const int k = s_nmodels[a];
                if (k < 0) {                                     // getSubset retries; gives up after max_attempts
                    if (++failed_attempts >= max_attempts) s_done = 1;
                    continue;
                }
                failed_attempts = 0;
                for (int r = 0; r < k; r++) {
                    if (!lmeds) {
                        const int good = (int)s_score[a][r];
                        if (good > (max_good > FM_MODEL_POINTS - 1 ? max_good : FM_MODEL_POINTS - 1)) {
                            max_good = good; best_slot = a; best_root = r; found = true;
                            niters = fm_update_iters(0.99, (double)(m - good) / m, FM_MODEL_POINTS, niters);
                        }
                    } else if ((double)s_score[a][r] < s_min_median) {
                        s_min_median = (double)s_score[a][r]; best_slot = a; best_root = r; found = true;
                    }
                }
                iter++;
            }
            if (iter >= niters) s_done = 1;
            s_best_slot = best_slot; s_best_root = best_root; s_found = found ? 1 : 0;
        }
        __syncthreads();
        if (s_best_slot >= 0 && tid < 9) s_best[tid] = models[27 * s_best_slot + 9 * s_best_root + tid];
        __syncthreads();          // s_best is taken before the next chunk overwrites the model scratch
        if (s_done) break;
        chunk = chunk * 4 < RF_THREADS ? chunk * 4 : RF_THREADS;
    }
    // no model (OpenCV returns an empty mask): every survivor is kept
    if (!s_found) return;
    float t = t_ransac;
    if (lmeds) {
        double sigma = 2.5 * 1.4826 * (1 + 5. / (m - FM_MODEL_POINTS)) * sqrt(s_min_median);
        if (sigma < 0.001) sigma = 0.001;
        t = (float)(sigma * sigma);
    }
    for (int j = tid; j < m; j += RF_THREADS)
        if (!(fm_error(s_best, m1[j], m2[j]) <= t)) S.status[o + src[j]] = 0;
}

}  // namespace

size_t reject_with_f_models(int n_sets) { return (size_t)n_sets * RF_THREADS * 27; }

int launch_reject_with_f_step(const PointSetArrays& S, int n_sets, int cap, const CamParams* d_cams, const uint8_t* d_lane, int W, int H,
                              double threshold, double* d_models, cudaStream_t st) {
    if (n_sets <= 0) return DVFE_OK;
    const size_t smem = (size_t)cap * (2 * sizeof(float2) + sizeof(unsigned short));
    DVFE_LAUNCH(k_reject_with_f_step, n_sets, RF_THREADS, smem, st, S, cap, d_cams, d_lane, W / 2.0, H / 2.0, threshold, d_models);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}
