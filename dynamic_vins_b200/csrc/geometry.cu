// Epipolar outlier rejection and the dense extra-point sampler of dynamic mode (SURVEY §8f N4):
//   InstsFeatManager::RejectWithF   dynamic_vins/src/front_end/dynamic_tracker.cpp:831-849
//   FeatureTracker::RejectWithF     dynamic_vins/src/front_end/background_tracker.cpp:520-550 (same call, commented out there)
//   InstFeat::DetectExtraPoints     dynamic_vins/src/front_end/instance_feature.cpp:413-461
//
// RejectWithF = liftProjective of both point lists (fp64), re-projection with kFocalLength = 460 about the image centre,
// narrowing to float, then cv::findFundamentalMat(cur, prev, FM_RANSAC, F_threshold, 0.99, status).  OpenCV
// (modules/calib3d/src/{fundam,ptsetreg}.cpp) runs that as a SEQUENTIAL loop: draw a 7-point sample from cv::RNG(-1), solve the
// cubic of the 7-point algorithm (up to 3 models), count the inliers of each over all points, keep the best and shorten the
// loop from the inlier ratio (8 <= n < 15: LMedS, the model with the smallest median error).  Which sample is drawn at iteration
// k depends only on the RNG and the point coordinates, never on the models, so the loop splits into
//   (a) one thread replaying the RNG: a chunk of candidate samples (index 7-tuples),
//   (b) one thread per candidate sample: collinearity test, 7-point solve, inlier count / median of every root over all points,
//   (c) one thread replaying OpenCV's bookkeeping over the chunk in sample order (best model, iteration budget, give-up rule),
// repeated until (c) says the sequential loop would have stopped.  One CTA per problem; all arithmetic in fp64 without
// contraction (-fmad=false) in the operation order of the OpenCV source, so the status bytes equal the CPU loop's.
#include "fm.cuh"
#include "kernels.cuh"
#include "tracker.h"

#define DVFE_CHECK(call)                  \
    do {                                  \
        int rc__ = (call);                \
        if (rc__ != DVFE_OK) return rc__; \
    } while (0)

#define FM_THREADS 256          // candidate samples per chunk = threads per CTA

namespace {

struct FmProblem {
    const float2* cur;       // distorted pixel positions, current frame  (findFundamentalMat's points1 after undistortion)
    const float2* prev;      // ... previous frame                         (points2)
    float2* un;              // scratch: 2 n undistorted / re-projected points (cur then prev)
    double* models;          // scratch: FM_THREADS * 27 doubles
    uint8_t* status;         // out: n bytes
    int n;
};

// One CTA per problem.
__global__ void __launch_bounds__(FM_THREADS) k_reject_with_f(const FmProblem* __restrict__ problems, CamParams cam, double half_col,
                                                             double half_row, double threshold, double confidence) {
    __shared__ int s_idx[FM_THREADS][FM_MODEL_POINTS];
    __shared__ int s_nmodels[FM_THREADS];            // -1: sample rejected (collinear), else number of roots
    __shared__ double s_score[FM_THREADS][3];        // RANSAC: inlier count; LMedS: median error
    __shared__ int s_done, s_found, s_best_slot, s_best_root;
    __shared__ double s_best[9], s_min_median;
    const FmProblem P = problems[blockIdx.x];
    const int n = P.n, tid = threadIdx.x;
    if (n < 7) return;                               // no model: the caller reports an empty status

    // undistort + re-project with the virtual focal length (float, as cv::Point2f((float)x, (float)y))
    for (int i = tid; i < 2 * n; i += FM_THREADS) P.un[i] = fm_reproject(cam, i < n ? P.cur[i] : P.prev[i - n], half_col, half_row);
    if (n == 7) {                                    // the solver runs once and the mask is set to all ones
        if (tid < 7) P.status[tid] = 1;
        return;
    }
    __syncthreads();
    const float2* __restrict__ m1 = P.un;
    const float2* __restrict__ m2 = P.un + n;
    const bool lmeds = n < 15;
    const float t_ransac = (float)(threshold * threshold);

    // thread 0 carries the sequential state of the OpenCV loop
    FmRng rng{~0ull};
    int niters = FM_MAX_ITERS, iter = 0, max_good = 0, failed_attempts = 0;
    bool found = false;
    if (tid == 0) {
        s_done = 0; s_min_median = 1.7976931348623157e308;
        if (lmeds) { niters = fm_update_iters(confidence, 0.45, FM_MODEL_POINTS, FM_MAX_ITERS); if (niters < 3) niters = 3; }
    }
    const int max_attempts = lmeds ? 1000 : 10000;   // getSubset's give-up bound per iteration
    double* my_models = P.models + (size_t)tid * 27;

    for (;;) {
        // (a) the RNG stream: FM_THREADS candidate samples, duplicates inside a sample redrawn
        if (tid == 0) {
            for (int a = 0; a < FM_THREADS; a++)
                for (int i = 0; i < FM_MODEL_POINTS; i++) {
                    int v;
                    bool dup;
                    do {
                        v = rng.uniform(0, n);
                        dup = false;
                        for (int j = 0; j < i; j++) dup |= s_idx[a][j] == v;
                    } while (dup);
                    s_idx[a][i] = v;
                }
        }
        __syncthreads();
        // (b) one candidate sample per thread
        {
            int idx[7];
            for (int i = 0; i < 7; i++) idx[i] = s_idx[tid][i];
            int k = -1;
            if (!fm_collinear(m1, idx) && !fm_collinear(m2, idx)) {
                double F[27];
                k = fm_run7(m1, m2, idx, F);
                for (int r = 0; r < k; r++) {
                    const double* Fr = F + 9 * r;
                    if (!lmeds) {
                        int good = 0;
                        for (int j = 0; j < n; j++) good += fm_error(Fr, m1[j], m2[j]) <= t_ransac;
                        s_score[tid][r] = (double)good;
                    } else {
                        float e[14];
                        for (int j = 0; j < n; j++) {            // insertion sort, n <= 14
                            const float v = fm_error(Fr, m1[j], m2[j]);
                            int q = j;
                            while (q > 0 && e[q - 1] > v) { e[q] = e[q - 1]; q--; }
                            e[q] = v;
                        }
                        s_score[tid][r] = (double)e[n / 2];       // std::nth_element(..., count / 2)
                    }
                    for (int q = 0; q < 9; q++) my_models[9 * r + q] = Fr[q];
                }
            }
            s_nmodels[tid] = k;
        }
        __syncthreads();
        // (c) OpenCV's loop bookkeeping replayed over the chunk in sample order
        if (tid == 0) {
            int best_slot = -1, best_root = 0;
            for (int a = 0; a < FM_THREADS && !s_done; a++) {
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
                            niters = fm_update_iters(confidence, (double)(n - good) / n, FM_MODEL_POINTS, niters);
                        }
                    } else if (s_score[a][r] < s_min_median) {
                        s_min_median = s_score[a][r]; best_slot = a; best_root = r; found = true;
                    }
                }
                iter++;
            }
            if (iter >= niters) s_done = 1;
            s_best_slot = best_slot; s_best_root = best_root; s_found = found ? 1 : 0;
        }
        __syncthreads();
        if (s_best_slot >= 0 && tid < 9) s_best[tid] = P.models[(size_t)s_best_slot * 27 + 9 * s_best_root + tid];
        __syncthreads();          // s_best is taken before the next chunk overwrites the model scratch
        if (s_done) break;
    }
    if (!s_found) {                // no model: OpenCV leaves the mask unwritten; reported as all zero
        for (int j = tid; j < n; j += FM_THREADS) P.status[j] = 0;
        return;
    }
    float t = t_ransac;
    if (lmeds) {
        double sigma = 2.5 * 1.4826 * (1 + 5. / (n - FM_MODEL_POINTS)) * sqrt(s_min_median);
        if (sigma < 0.001) sigma = 0.001;
        t = (float)(sigma * sigma);
    }
    for (int j = tid; j < n; j += FM_THREADS) P.status[j] = fm_error(s_best, m1[j], m2[j]) <= t ? 1 : 0;
}

// InstFeat::DetectExtraPoints: one thread per grid sample, order-preserving compaction (row-major sample order) by a block scan
struct ExtraJob {
    const uint8_t* mask;     // ROI mask, rows x cols
    int mask_pitch;
    int rows, cols;
    int box_x, box_y;        // box2d->rect.tl()
    double* out;             // 3 doubles per point
    int* n_out;
};

__global__ void __launch_bounds__(256) k_detect_extra_points(const ExtraJob* __restrict__ jobs, const float* __restrict__ disp, int disp_pitch,
                                                              float fx, float fy, float cx, float cy, float baseline) {
    __shared__ int s_warp[8];
    __shared__ int s_base;
    const ExtraJob J = jobs[blockIdx.x];
    const int step = (int)fmax(sqrt(0.8 * J.rows * J.cols / 1000.), 2.);
    const int gw = (J.cols + step - 1) / step, gh = (J.rows + step - 1) / step, total = gw * gh;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int base = 0; base < total; base += 256) {
        const int s = base + tid;
        bool keep = false;
        float x3 = 0.f, y3 = 0.f, depth = 0.f;
        if (s < total) {
            const int i = (s / gw) * step, j = (s - (s / gw) * gw) * step;
            if (J.mask[(size_t)i * J.mask_pitch + j] > 0) {
                const int r = i + J.box_y, c = j + J.box_x;
                const float d = disp[(size_t)r * disp_pitch + c];
                if (d > 0.f && d == d) {
                    depth = fx * baseline / d;
                    if (!((double)depth <= 0.1 || depth > 100.f)) {
                        x3 = ((float)c - cx) * depth / fx;
                        y3 = ((float)r - cy) * depth / fy;
                        keep = true;
                    }
                }
            }
        }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        int off = s_base;
        for (int w = 0; w < warp; w++) off += s_warp[w];
        off += __popc(bal & ((1u << lane) - 1u));
        if (keep) { J.out[3 * (size_t)off] = x3; J.out[3 * (size_t)off + 1] = y3; J.out[3 * (size_t)off + 2] = depth; }
        __syncthreads();
        if (tid == 0) { int t = 0; for (int w = 0; w < 8; w++) t += s_warp[w]; s_base += t; }
        __syncthreads();
    }
    if (tid == 0) *J.n_out = s_base;
}

struct DevMem {
    void* p = nullptr;
    ~DevMem() { if (p) cudaFree(p); }
    int alloc(size_t bytes) {
        DVFE_CUDA(cudaMalloc(&p, bytes ? bytes : 1));
        return DVFE_OK;
    }
    template <typename T> T* as() { return reinterpret_cast<T*>(p); }
};

int need_device() {
    int count = 0;
    const cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0) {
        dvfe_set_error("no CUDA device available (%s): libdvfe has no CPU fallback", cudaGetErrorString(e));
        return DVFE_ERR_NO_DEVICE;
    }
    return DVFE_OK;
}
}  // namespace

extern "C" int dvfe_op_reject_with_f(const dvfe_camera* cam, const float* cur_pts, const float* prev_pts, int n, int col, int row,
                                     double f_threshold, uint8_t* status, int* n_status) {
    if (!cam || n < 0 || !n_status || (n > 0 && (!cur_pts || !prev_pts || !status))) {
        dvfe_set_error("op_reject_with_f: bad argument");
        return DVFE_ERR_INVALID;
    }
    DVFE_CHECK(need_device());
    *n_status = 0;
    if (n < 7) return DVFE_OK;                       // cv::findFundamentalMat returns an empty matrix and leaves `status` empty
    DevMem d_cur, d_prev, d_un, d_models, d_status, d_prob;
    DVFE_CHECK(d_cur.alloc(sizeof(float2) * n));
    DVFE_CHECK(d_prev.alloc(sizeof(float2) * n));
    DVFE_CHECK(d_un.alloc(sizeof(float2) * 2 * n));
    DVFE_CHECK(d_models.alloc(sizeof(double) * 27 * FM_THREADS));
    DVFE_CHECK(d_status.alloc(n));
    DVFE_CHECK(d_prob.alloc(sizeof(FmProblem)));
    DVFE_CUDA(cudaMemcpy(d_cur.p, cur_pts, sizeof(float2) * n, cudaMemcpyHostToDevice));
    DVFE_CUDA(cudaMemcpy(d_prev.p, prev_pts, sizeof(float2) * n, cudaMemcpyHostToDevice));
    FmProblem P{d_cur.as<float2>(), d_prev.as<float2>(), d_un.as<float2>(), d_models.as<double>(), d_status.as<uint8_t>(), n};
    DVFE_CUDA(cudaMemcpy(d_prob.p, &P, sizeof(P), cudaMemcpyHostToDevice));
    double thr = f_threshold;
    if (thr <= 0) thr = 3;                           // cv::findFundamentalMat: param1 <= 0 -> 3
    DVFE_LAUNCH(k_reject_with_f, 1, FM_THREADS, 0, 0, d_prob.as<FmProblem>(), make_cam(*cam), col / 2.0, row / 2.0, thr, 0.99);
    DVFE_CUDA(cudaGetLastError());
    DVFE_CUDA(cudaDeviceSynchronize());
    DVFE_CUDA(cudaMemcpy(status, d_status.p, n, cudaMemcpyDeviceToHost));
    *n_status = n;
    return DVFE_OK;
}

extern "C" int dvfe_op_detect_extra_points(const uint8_t* roi_mask, int rows, int cols, int mask_pitch, const float* disp, int disp_w,
                                           int disp_h, int disp_pitch, int box_x, int box_y, float fx, float fy, float cx, float cy,
                                           float baseline, double* out, int cap, int* n_out) {
    if (!roi_mask || !disp || !out || !n_out || rows < 1 || cols < 1 || mask_pitch < cols || disp_pitch < disp_w || box_x < 0 || box_y < 0 ||
        box_x + cols > disp_w || box_y + rows > disp_h) {
        dvfe_set_error("op_detect_extra_points: bad argument (the box must lie inside the disparity map)");
        return DVFE_ERR_INVALID;
    }
    DVFE_CHECK(need_device());
    const int step = (int)fmax(sqrt(0.8 * rows * cols / 1000.), 2.);
    const int total = ((cols + step - 1) / step) * ((rows + step - 1) / step);
    DevMem d_mask, d_disp, d_out, d_n, d_job;
    DVFE_CHECK(d_mask.alloc((size_t)rows * cols));
    DVFE_CHECK(d_disp.alloc(sizeof(float) * (size_t)disp_w * disp_h));
    DVFE_CHECK(d_out.alloc(sizeof(double) * 3 * total));
    DVFE_CHECK(d_n.alloc(sizeof(int)));
    DVFE_CHECK(d_job.alloc(sizeof(ExtraJob)));
    DVFE_CUDA(cudaMemcpy2D(d_mask.p, cols, roi_mask, mask_pitch, cols, rows, cudaMemcpyHostToDevice));
    DVFE_CUDA(cudaMemcpy2D(d_disp.p, sizeof(float) * disp_w, disp, sizeof(float) * disp_pitch, sizeof(float) * disp_w, disp_h,
                           cudaMemcpyHostToDevice));
    ExtraJob J{d_mask.as<uint8_t>(), cols, rows, cols, box_x, box_y, d_out.as<double>(), d_n.as<int>()};
    DVFE_CUDA(cudaMemcpy(d_job.p, &J, sizeof(J), cudaMemcpyHostToDevice));
    DVFE_LAUNCH(k_detect_extra_points, 1, 256, 0, 0, d_job.as<ExtraJob>(), d_disp.as<float>(), disp_w, fx, fy, cx, cy, baseline);
    DVFE_CUDA(cudaGetLastError());
    DVFE_CUDA(cudaDeviceSynchronize());
    int n = 0;
    DVFE_CUDA(cudaMemcpy(&n, d_n.p, sizeof(int), cudaMemcpyDeviceToHost));
    *n_out = n;
    if (n > cap) {
        dvfe_set_error("op_detect_extra_points: %d points do not fit the output capacity %d", n, cap);
        return DVFE_ERR_CAPACITY;
    }
    DVFE_CUDA(cudaMemcpy(out, d_out.p, sizeof(double) * 3 * n, cudaMemcpyDeviceToHost));
    return DVFE_OK;
}
