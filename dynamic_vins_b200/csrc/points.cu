// Per-point bookkeeping kernels — replace the std::vector / std::map glue of InstFeat
// (dynamic_vins/src/front_end/instance_feature.{h,cpp}) and FeatureTracker::SetOutputFeats:
//   ReduceVector (front_end/feature_utils.h:77-85)            -> order-preserving compaction
//   InstFeat::UndistortedPts / RightUndistortedPts / UndistortedPointsWithAddOffset
//     (instance_feature.cpp:94-103,123-133,137-146) -> PinholeCamera::liftProjective
//     (/root/reference/camera_models/src/camera_models/PinholeCamera.cc:450-510, distortion :646-660), fp64
//   InstFeat::PtsVelocity / RightPtsVelocity (instance_feature.cpp:26-85): the id->point maps are replaced by
//     values carried with the points through the compaction (an id is in prev_id_pts iff the point existed in
//     the previous frame)
//   InstFeat::PostProcess (instance_feature.h:88-101): prev := curr, done in place
//   FeatureTracker::SetOutputFeats (front_end/background_tracker.cpp:340-392): records sorted by (id, cam)
#include "kernels.cuh"
#include "state.cuh"

CamParams make_cam(const dvfe_camera& c) {
    CamParams p;
    p.inv_K11 = 1.0 / c.fx;
    p.inv_K13 = -c.cx / c.fx;
    p.inv_K22 = 1.0 / c.fy;
    p.inv_K23 = -c.cy / c.fy;
    p.k1 = c.k1; p.k2 = c.k2; p.p1 = c.p1; p.p2 = c.p2;
    p.no_distortion = (c.k1 == 0.0 && c.k2 == 0.0 && c.p1 == 0.0 && c.p2 == 0.0);
    return p;
}

__device__ __forceinline__ float2 lift_projective(const CamParams& cam, float px, float py) {
    const double u = (double)px, v = (double)py;
    const double mx_d = cam.inv_K11 * u + cam.inv_K13;
    const double my_d = cam.inv_K22 * v + cam.inv_K23;
    double mx_u = mx_d, my_u = my_d;
    if (!cam.no_distortion) {
#pragma unroll 1
        for (int i = 0; i < 8; i++) {      // n = 8 fixed-point steps, the first from (mx_d, my_d)
            const double x = mx_u, y = my_u;
            const double mx2 = x * x, my2 = y * y, mxy = x * y;
            const double rho2 = mx2 + my2;
            const double rad = cam.k1 * rho2 + cam.k2 * rho2 * rho2;
            const double dux = x * rad + 2.0 * cam.p1 * mxy + cam.p2 * (rho2 + 2.0 * mx2);
            const double duy = y * rad + 2.0 * cam.p2 * mxy + cam.p1 * (rho2 + 2.0 * my2);
            mx_u = mx_d - dux;
            my_u = my_d - duy;
        }
    }
    return make_float2((float)mx_u, (float)my_u);    // b.x / b.z with b.z == 1.0
}

__global__ void k_lift(CamParams cam, const float2* __restrict__ pts, int n, float offx, float offy, float2* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float2 p = pts[i];
    out[i] = lift_projective(cam, p.x + offx, p.y + offy);
}

int launch_lift(const CamParams& cam, const float2* pts, int n, float offx, float offy, float2* out, cudaStream_t st) {
    if (n <= 0) return DVFE_OK;
    DVFE_LAUNCH(k_lift, (n + 127) / 128, 128, 0, st, cam, pts, n, offx, offy, out);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

// ---- ReduceVector after the temporal LK: keep status != 0, preserve order; track_cnt++ ---------------
// One block per point set; in-place (destination index <= source index, chunks are read before written).
// old_idx (nullable): old_idx[set*cap + j] = the index the survivor at j had before the compaction, -1 for the free slots behind
// the survivors (the points the detection appends there are new): lets the stereo LK pick up the templates the temporal LK's
// backward pass built for the same point.
__global__ void __launch_bounds__(256) k_compact_tracked(PointSetArrays S, int cap, const uint8_t* __restrict__ active,
                                                         int* __restrict__ old_idx) {
    __shared__ int s_warp[8];
    __shared__ int s_base;
    const int set = blockIdx.x;
    if (active != nullptr && !active[set]) return;      // TrackLeft was not called for this set
    const size_t o = (size_t)set * cap;
    const int n = S.n[set];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int c0 = 0; c0 < n; c0 += 256) {
        const int i = c0 + tid;
        const bool keep = (i < n) && S.status[o + i] != 0;
        float2 p = make_float2(0, 0), un = p, rp = p;
        uint32_t id = 0; int32_t tc = 0; uint8_t rv = 0;
        if (keep) {
            p = S.lk_out[o + i]; un = S.un[o + i]; id = S.ids[o + i]; tc = S.track_cnt[o + i];
            rp = S.rprev_un[o + i]; rv = S.rprev_valid[o + i];
        }
        const unsigned ballot = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[warp] = __popc(ballot);
        __syncthreads();
        int off = s_base;
        for (int wv = 0; wv < warp; wv++) off += s_warp[wv];
        if (keep) {
            const int j = off + __popc(ballot & ((1u << lane) - 1));
            S.pts[o + j] = p; S.un[o + j] = un; S.ids[o + j] = id; S.track_cnt[o + j] = tc + 1;
            S.rprev_un[o + j] = rp; S.rprev_valid[o + j] = rv;
            if (old_idx != nullptr) old_idx[o + j] = i;
        }
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int wv = 0; wv < 8; wv++) tot += s_warp[wv];
            s_base += tot;
        }
        __syncthreads();
    }
    if (old_idx != nullptr)
        for (int j = s_base + tid; j < cap; j += 256) old_idx[o + j] = -1;
    if (tid == 0) S.n[set] = s_base;
}

int launch_compact(const PointSetArrays& S, int n_sets, int cap, cudaStream_t st, const uint8_t* d_active, int* d_old_idx) {
    if (n_sets <= 0) return DVFE_OK;
    DVFE_LAUNCH(k_compact_tracked, n_sets, 256, 0, st, S, cap, d_active, d_old_idx);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

// ---- UndistortedPts + PtsVelocity for the left image; un[] holds prev_id_pts on entry, curr on exit ------
__global__ void __launch_bounds__(128) k_left_post(PointSetArrays S, int cap, CamParams cam, const double* __restrict__ dt,
                                                   const float2* __restrict__ offset /* nullable, per set */,
                                                   const uint8_t* __restrict__ active) {
    const int set = blockIdx.y;
    if (active != nullptr && !active[set]) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S.n[set]) return;
    const size_t k = (size_t)set * cap + i;
    const float2 p = S.pts[k];
    const float2 off = offset ? offset[set] : make_float2(0.f, 0.f);
    const float2 un = lift_projective(cam, p.x + off.x, p.y + off.y);
    float2 vel = make_float2(0.f, 0.f);
    if (S.track_cnt[k] > 1) {          // id is in prev_id_pts  <=>  the point was tracked from the last frame
        const float2 prev = S.un[k];
        const double d = dt[set];
        vel.x = (float)((double)(un.x - prev.x) / d);
        vel.y = (float)((double)(un.y - prev.y) / d);
    } else {
        S.rprev_valid[k] = 0;          // a new id has no entry in right_prev_id_pts
    }
    S.un[k] = un;
    S.vel[k] = vel;
}

int launch_left_post(const PointSetArrays& S, int n_sets, int cap, const CamParams& cam, const double* d_dt,
                     const float2* d_offset, cudaStream_t st, const uint8_t* d_active) {
    if (n_sets <= 0) return DVFE_OK;
    dim3 grid((cap + 127) / 128, n_sets);
    DVFE_LAUNCH(k_left_post, grid, 128, 0, st, S, cap, cam, d_dt, d_offset, d_active);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

// ---- right image: RightUndistortedPts + RightPtsVelocity + SetOutputFeats --------------------------------
// One block per point set.  Emits dvfe_obs records sorted by (id, cam): the point arrays are always in
// ascending id order (survivors keep their order, new ids are appended).
// lanes (nullable, per set): 0 = the set had no frame in this step (no records, nothing written), else LANE_PRESENT and
// LANE_STEREO when it had a right image; null = every set present, with a right image iff stereo_now.
__global__ void __launch_bounds__(256) k_right_post_pack(PointSetArrays S, int cap, CamParams cam1, const double* __restrict__ dt,
                                                         int stereo_all, const uint8_t* __restrict__ lanes,
                                                         dvfe_obs* __restrict__ obs, int* __restrict__ n_obs) {
    __shared__ int s_warp[8];
    __shared__ int s_base;
    const int set = blockIdx.x;
    if (lanes != nullptr && lanes[set] == 0) {
        if (threadIdx.x == 0) n_obs[set] = 0;
        return;
    }
    const int stereo_now = lanes != nullptr ? (lanes[set] & LANE_STEREO) != 0 : stereo_all;
    const size_t o = (size_t)set * cap;
    const int n = S.n[set];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    dvfe_obs* out = obs + (size_t)set * 2 * cap;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int c0 = 0; c0 < n; c0 += 256) {
        const int i = c0 + tid;
        const bool has_r = stereo_now && (i < n) && S.rstatus[o + i] != 0;
        float2 run = make_float2(0, 0), rvel = run, rp = run;
        if (has_r) {
            rp = S.rpts[o + i];
            run = lift_projective(cam1, rp.x, rp.y);
            if (S.rprev_valid[o + i]) {
                const float2 prev = S.rprev_un[o + i];
                const double d = dt[set];
                rvel.x = (float)((double)(run.x - prev.x) / d);
                rvel.y = (float)((double)(run.y - prev.y) / d);
            }
        }
        if (stereo_now && i < n) {     // right_prev_id_pts = right_curr_id_pts
            S.rprev_valid[o + i] = has_r ? 1 : 0;
            if (has_r) S.rprev_un[o + i] = run;
        }
        const unsigned ballot = __ballot_sync(0xffffffffu, has_r);
        if (lane == 0) s_warp[warp] = __popc(ballot);
        __syncthreads();
        int off = s_base;
        for (int wv = 0; wv < warp; wv++) off += s_warp[wv];
        if (i < n) {
            const int j = i + off + __popc(ballot & ((1u << lane) - 1));
            const float2 p = S.pts[o + i], un = S.un[o + i], vel = S.vel[o + i];
            dvfe_obs r;
            r.id = S.ids[o + i]; r.cam = 0;
            r.v[0] = un.x; r.v[1] = un.y; r.v[2] = 1.0; r.v[3] = p.x; r.v[4] = p.y; r.v[5] = vel.x; r.v[6] = vel.y;
            out[j] = r;
            if (has_r) {
                r.cam = 1;
                r.v[0] = run.x; r.v[1] = run.y; r.v[3] = rp.x; r.v[4] = rp.y; r.v[5] = rvel.x; r.v[6] = rvel.y;
                out[j + 1] = r;
            }
        }
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int wv = 0; wv < 8; wv++) tot += s_warp[wv];
            s_base += tot;
        }
        __syncthreads();
    }
    if (tid == 0) n_obs[set] = n + s_base;
}

int launch_right_post_pack(const PointSetArrays& S, int n_sets, int cap, const CamParams& cam1, const double* d_dt,
                           int stereo_now, dvfe_obs* obs, int* n_obs, cudaStream_t st, const uint8_t* d_lane) {
    if (n_sets <= 0) return DVFE_OK;
    DVFE_LAUNCH(k_right_post_pack, n_sets, 256, 0, st, S, cap, cam1, d_dt, stereo_now, d_lane, obs, n_obs);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

// ---- instances: RightUndistortedPts + RightPtsVelocity + InstsFeatManager::Output record -----------------------
// (front_end/dynamic_tracker.cpp:462-471, 521-577).  One record per point at out[set*cap + i]; ids ascend with i.
// lanes (nullable, per set): whether the set's stream had a right image (LANE_STEREO) in place of stereo_all for every set.
__global__ void __launch_bounds__(128) k_inst_post_pack(PointSetArrays S, int cap, CamParams cam1, const double* __restrict__ dt,
                                                        const uint8_t* __restrict__ active, int stereo_all,
                                                        const uint8_t* __restrict__ lanes, const uint32_t* __restrict__ inst_id,
                                                        dvfe_inst_obs* __restrict__ out, int* __restrict__ n_out) {
    const int set = blockIdx.y;
    if (!active[set]) return;
    const int stereo_now = lanes != nullptr ? (lanes[set] & LANE_STEREO) != 0 : stereo_all;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    // the record count of this call, snapshotted into the call's own buffer: S.n is rewritten by the next step while the
    // download stream may still be reading
    if (i == 0) n_out[set] = S.n[set];
    if (i >= S.n[set]) return;
    const size_t k = (size_t)set * cap + i;
    const bool has_r = stereo_now && S.rstatus[k] != 0;
    float2 run = make_float2(0, 0), rvel = run;
    if (has_r) {
        const float2 rp = S.rpts[k];
        run = lift_projective(cam1, rp.x, rp.y);
        if (S.rprev_valid[k]) {
            const float2 prev = S.rprev_un[k];
            const double d = dt[set];
            rvel.x = (float)((double)(run.x - prev.x) / d);
            rvel.y = (float)((double)(run.y - prev.y) / d);
        }
    }
    if (stereo_now) {      // right_prev_id_pts = right_curr_id_pts (PostProcess)
        S.rprev_valid[k] = has_r ? 1 : 0;
        if (has_r) S.rprev_un[k] = run;
    }
    const float2 p = S.pts[k], un = S.un[k], vel = S.vel[k];
    dvfe_inst_obs r;
    r.inst_id = inst_id[set]; r.id = S.ids[k]; r.is_stereo = has_r ? 1 : 0; r.reserved = 0;
    r.point[0] = un.x; r.point[1] = un.y; r.point[2] = 1.0;
    r.vel[0] = vel.x; r.vel[1] = vel.y;
    r.point_right[0] = has_r ? (double)run.x : 0.0; r.point_right[1] = has_r ? (double)run.y : 0.0;
    r.point_right[2] = has_r ? 1.0 : 0.0;
    r.vel_right[0] = has_r ? (double)rvel.x : 0.0; r.vel_right[1] = has_r ? (double)rvel.y : 0.0;
    r.uv[0] = p.x; r.uv[1] = p.y;
    r.disp = 0.0;
    out[k] = r;
}

int launch_inst_post_pack(const PointSetArrays& S, int n_sets, int cap, const CamParams& cam1, const double* d_dt,
                          const uint8_t* d_active, int stereo_now, const uint8_t* d_lane, const uint32_t* d_inst_id,
                          dvfe_inst_obs* out, int* d_n_out, cudaStream_t st) {
    if (n_sets <= 0) return DVFE_OK;
    dim3 grid((cap + 127) / 128, n_sets);
    DVFE_LAUNCH(k_inst_post_pack, grid, 128, 0, st, S, cap, cam1, d_dt, d_active, stereo_now, d_lane, d_inst_id, out, d_n_out);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

// n[set] = 0 for the flagged sets (InstsFeatManager::ClearState, front_end/dynamic_tracker.cpp:41-58)
__global__ void k_clear_sets(int* n, const uint8_t* __restrict__ flags, int n_sets) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_sets && flags[i]) n[i] = 0;
}

int launch_clear_sets(int* d_n, const uint8_t* d_flags, int n_sets, cudaStream_t st) {
    if (n_sets <= 0) return DVFE_OK;
    DVFE_LAUNCH(k_clear_sets, (n_sets + 127) / 128, 128, 0, st, d_n, d_flags, n_sets);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}
