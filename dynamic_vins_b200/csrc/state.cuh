// Device-resident tracker state (replaces the std::vector / std::map members of InstFeat,
// dynamic_vins/src/front_end/instance_feature.h:103-137).  Struct of arrays, `cap` slots per point set.
#pragma once
#include "common.cuh"

struct PointSetArrays {
    float2* pts;            // curr_points (== last_points between frames)
    float2* lk_out;         // temporal LK result before compaction
    float2* un;             // prev_id_pts values on entry of a frame, curr_un_points on exit
    float2* vel;            // pts_velocity
    uint32_t* ids;
    int32_t* track_cnt;
    uint8_t* status;        // temporal LK status
    float2* rpts;           // right_points, indexed like pts (valid where rstatus)
    uint8_t* rstatus;       // stereo LK status of this frame
    float2* rprev_un;       // right_prev_id_pts values
    uint8_t* rprev_valid;   // id present in right_prev_id_pts
    int* n;                 // [n_sets]
};

int launch_compact(const PointSetArrays& S, int n_sets, int cap, cudaStream_t st, const uint8_t* d_active = nullptr,
                   int* d_old_idx = nullptr);
struct CamParams;
int launch_left_post(const PointSetArrays& S, int n_sets, int cap, const CamParams& cam, const double* d_dt,
                     const float2* d_offset, cudaStream_t st, const uint8_t* d_active = nullptr);
int launch_inst_post_pack(const PointSetArrays& S, int n_sets, int cap, const CamParams& cam1, const double* d_dt,
                          const uint8_t* d_active, int stereo_now, const uint8_t* d_lane, const uint32_t* d_inst_id,
                          dvfe_inst_obs* out, int* d_n_out, cudaStream_t st);
int launch_clear_sets(int* d_n, const uint8_t* d_flags, int n_sets, cudaStream_t st);
int launch_right_post_pack(const PointSetArrays& S, int n_sets, int cap, const CamParams& cam1, const double* d_dt,
                           int stereo_now, dvfe_obs* obs, int* n_obs, cudaStream_t st, const uint8_t* d_lane = nullptr);
