// Shared device/host definitions for the dvfe kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/dvfe.h"
#include "../../include/dvfe/reject_with_f.h"

// Padded pyramid storage.  LK reads a 22x22 window whose origin lies in [-21, w-1] x [-21, h-1]
// (cv::calcOpticalFlowPyrLK keeps a winSize border around every level), plus one more pixel for
// the on-the-fly Scharr taps, so every level is stored with a REFLECT_101 border of PADX/PADY
// pixels; rows start 16-byte aligned so the LK gather can use aligned word loads.
#define DVFE_PADX 32
#define DVFE_PADY 24
#define DVFE_WIN 21
#define DVFE_HALF_WIN 10.0f

struct PyrLevel {
    int w, h;          // level size
    int pitch;         // bytes per padded row (multiple of 16, >= w + 2*PADX)
    unsigned offset;   // byte offset of padded row 0 inside the pyramid allocation
};
struct PyrDesc {
    int n_levels;      // levels kept = effective maxLevel + 1 (cv::buildOpticalFlowPyramid truncation rule)
    PyrLevel lv[DVFE_MAX_PYR_LEVELS];
    unsigned bytes;    // size of one pyramid (multiple of 256)
};

__host__ __device__ __forceinline__ int reflect101(int p, int n) {
    // cv::BORDER_REFLECT_101:  gfedcb|abcdefgh|gfedcba
    if (n == 1) return 0;
    while (p < 0 || p >= n) p = (p < 0) ? -p : 2 * (n - 1) - p;
    return p;
}

__host__ __device__ __forceinline__ const uint8_t* pyr_px(const uint8_t* base, const PyrLevel& L) {
    // pointer to pixel (0,0) of the level
    return base + L.offset + (size_t)DVFE_PADY * L.pitch + DVFE_PADX;
}

static inline PyrDesc make_pyr_desc(int w, int h, int max_level) {
    PyrDesc d{};
    unsigned off = 0;
    int lw = w, lh = h, l = 0;
    for (;;) {
        PyrLevel& L = d.lv[l];
        L.w = lw; L.h = lh;
        L.pitch = ((lw + 2 * DVFE_PADX) + 15) & ~15;
        L.offset = off;
        off += (unsigned)(((size_t)L.pitch * (lh + 2 * DVFE_PADY) + 255) & ~(size_t)255);
        l++;
        if (l > max_level || l >= DVFE_MAX_PYR_LEVELS) break;
        int nw = (lw + 1) / 2, nh = (lh + 1) / 2;
        if (nw <= DVFE_WIN || nh <= DVFE_WIN) break;   // buildOpticalFlowPyramid: stop when next level <= winSize
        lw = nw; lh = nh;
    }
    d.n_levels = l;
    // one pyramid = a whole number of level-0 rows, so a batch of pyramids is a pitched 3-D array whose slices
    // can be filled by a single cudaMemcpy3D straight from the caller's images
    const unsigned unit = (unsigned)d.lv[0].pitch * 16u;
    d.bytes = ((off + unit - 1) / unit) * unit;
    return d;
}

// ---- launch accounting / error handling -------------------------------------------------
extern unsigned long long g_dvfe_launches;
void dvfe_set_error(const char* fmt, ...);

#define DVFE_LAUNCH(kernel, grid, block, smem, stream, ...)            \
    do {                                                               \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);    \
        ++g_dvfe_launches;                                             \
    } while (0)

#define DVFE_CUDA(expr)                                                                       \
    do {                                                                                      \
        cudaError_t e__ = (expr);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            dvfe_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return DVFE_ERR_CUDA;                                                             \
        }                                                                                     \
    } while (0)

// ---- one independent point set processed by the LK kernel --------------------------------
// (a stream's background set, or one instance's ROI set)
struct LkGroup {
    const uint8_t* pyrA;     // pyramid of the template image (FeatureTrackByLK img1)
    const uint8_t* pyrB;     // pyramid of the search image   (FeatureTrackByLK img2)
    PyrDesc desc;            // geometry of both
    const float2* ptsA;      // pts1
    float2* ptsB;            // pts2 (out)
    float2* rev;             // backward-tracked pts1 (out, nullable)
    uint8_t* status;         // out
    const int* n;            // number of points (device)
    const uint8_t* mask;     // nullable: status &= mask[cvRound(pts2)] != 0
    int mask_pitch;
    float offx, offy;        // added to pts1 first (InstFeat::TrackRightByPad)
    unsigned* tcache;        // nullable: forward-pass template cache, LK_TCACHE_WORDS words per (point, level)
    unsigned* tcache_bwd;    // nullable: backward-pass template cache of the temporal call (same layout, indexed by the point's
                             // index in that call)
    const int* old_idx;      // nullable: per point, its index in the temporal call of this step (-1: new point)
};
// Template cache block of one (point, level): lane-major words, word j of lane l at [j * 32 + l]:
//   0..13  (Ix, Iy) int16 pairs of the lane's 14 window pixels;  14, 15  the lane's sum I*Ix, sum I*Iy;
//   16     lanes 0..2: A11, A12, A22 (float bits)
#define LK_TCACHE_WORDS (17 * 32)
#define LK_TCACHE_WRITE 1    // forward pass stores its templates (stereo call: template = current left image at the current points)
#define LK_TCACHE_READ 2     // forward pass loads them (next temporal call: same image, same points)
// The backward templates of the temporal call (current left image at the tracked positions, levels <= its backward maxLevel)
// are bit for bit the forward templates of the same step's stereo call at those levels for the points that survive:
#define LK_TCACHE_WRITE_BWD 4    // backward pass stores its templates in tcache_bwd (temporal call)
#define LK_TCACHE_READ_BWD 8     // forward pass loads levels <= reuse_max_level from tcache_bwd[old_idx] (stereo call)
