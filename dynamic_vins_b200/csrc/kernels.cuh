// Internal launch interfaces between the .cu files of libdvfe.
#pragma once
#include "common.cuh"

// A batch of images: set 0 (left) and set 1 (right), `per_set` images each, laid out with a stride.
struct PyrImgSet {
    const uint8_t* src[2];
    uint8_t* dst[2];
    size_t src_stride;   // bytes between consecutive source images of a set
    size_t dst_stride;   // bytes between consecutive pyramids of a set
    int per_set;
};

// job-based variants (per-instance ROIs have individual sizes)
struct PyrJob {
    const uint8_t* src;      // dense source image
    int sw, sh, spitch;      // its size; zero-extended to desc.lv[0]
    uint8_t* dst;            // pyramid allocation
    PyrDesc desc;
};
struct CropJob {
    const uint8_t* src;      // pixel (0,0) of the pitched source image
    int spitch;
    int x, y, w, h;
    uint8_t* dst;            // dense w x h
};
struct ErodeJob {
    const uint8_t* src;      // w x h at pitch `spitch`
    uint8_t* tmp;
    uint8_t* dst;
    int w, h, k;
    int spitch;
    int label_bit;           // < 0: src is the mask itself; >= 0: src is a label image, mask = bit `label_bit` set ? 255 : 0
};

// pyramid.cu
#define DVFE_L0_BUILD 0        // level 0 is copied from the source images (border included when pyr_level0_writes_border)
#define DVFE_L0_INTERIOR 1     // level 0's interior is already in place (DMA / ingest kernel), its border is not
#define DVFE_L0_COMPLETE 2     // level 0 is in place with its border
int launch_build_pyramids(const PyrImgSet& set, int n_img, const PyrDesc& desc, int spitch, cudaStream_t st,
                          int level0_mode = DVFE_L0_BUILD);
int launch_pyr_level0(const PyrImgSet& set, int n_img, const PyrDesc& desc, int spitch, cudaStream_t st);
bool pyr_level0_writes_border(const PyrDesc& desc);
// One image of a step's input, per stream (dvfe_track_frames): ptr == null = no image, nothing is read or written for it
struct ImgSrc {
    const uint8_t* ptr;
    int pitch;
};
// The gather form of launch_pyr_level0: image i is read at d_src[i] and written, border included when
// pyr_level0_writes_border, into level 0 of the pyramid at dst + i * dst_stride; absent images are not written
int launch_pyr_level0_table(const ImgSrc* d_src, uint8_t* dst, size_t dst_stride, int n_img, const PyrDesc& desc, cudaStream_t st);
// Frame ingest (prep.cu): optional fixed-point cv::remap (undistortion maps) + optional BGR -> gray, B images per launch,
// written at dst_pitch (straight into level 0 of a padded pyramid, or dense).
struct IngestArgs {
    const uint8_t* src;          // [B] images of `ch` interleaved channels
    size_t src_stride;           // bytes between images
    int src_pitch;
    int ch;                      // 1 (gray) | 3 (BGR)
    const short* map1;           // CV_16SC2 (x, y) per output pixel, dense w x h, or null = identity
    const unsigned short* map2;  // CV_16UC1 interpolation-table index (fy * 32 + fx), dense w x h
    uint8_t* dst;                // [B] gray images (ch_out = 1) or remapped `ch`-channel images (keep_channels)
    size_t dst_stride;
    int dst_pitch;
    int w, h, n_img;
    int keep_channels;           // 1: plain cv::remap of all channels (seam op); 0: output gray
};
// The maps of one image (per-stream undistortion): map1 == null = not remapped, only copied / converted to gray
struct IngestMaps {
    const short* map1;
    const unsigned short* map2;
};
// d_maps (nullable): [n_img] per-image maps in place of a.map1 / a.map2 (gray output only)
int launch_ingest(const IngestArgs& a, cudaStream_t st, const IngestMaps* d_maps = nullptr);
// The table form (gray output only): image i is read at d_src[i] (a.src / a.src_stride / a.src_pitch unused) and written at
// a.dst + i * a.dst_stride, remapped with d_maps[i] (nullable: a.map1 / a.map2 for every image); absent images are not written
int launch_ingest_table(const IngestArgs& a, const ImgSrc* d_src, cudaStream_t st, const IngestMaps* d_maps = nullptr);
// Dense copy of n_img images of `row` bytes x h rows: image i from d_src[i] to dst + i * dst_stride at dst_pitch; absent ones skipped
int launch_gather_images(const ImgSrc* d_src, uint8_t* dst, size_t dst_stride, int dst_pitch, int row, int h, int n_img,
                         cudaStream_t st);

int launch_build_pyramids_jobs(const PyrJob* d_jobs, int n_jobs, int max_w, int max_h, int max_levels, cudaStream_t st);
int launch_crop_jobs(const CropJob* d_jobs, int n_jobs, int max_w, int max_h, cudaStream_t st);
int launch_pyr_extract(const uint8_t* pyr, const PyrLevel& L, uint8_t* out, cudaStream_t st);
int launch_pyr_extract_bordered(const uint8_t* pyr, const PyrLevel& L, int border, uint8_t* out, cudaStream_t st);

// lk.cu
int launch_lk(const LkGroup* d_groups, int n_groups, int max_pts, int max_level, int flow_back, cudaStream_t st,
              int back_max_level = 1, double fb_threshold = 0.5, int tcache_flags = 0, int reuse_max_level = -1);

// gftt.cu
struct GfttJob {                 // one detection problem (a stream's image, or one instance ROI)
    const uint8_t* img;          // u8 image, pixel (0,0)
    int img_pitch;
    int w, h;
    int img_bordered;            // 1: img is pixel (0,0) of a padded pyramid level (REFLECT_101 border readable, rows 4-byte aligned)
    const uint8_t* region_mask;  // nullable (all 255)
    int region_pitch;
    uint8_t* mask;               // detection mask scratch (w x h, pitch mask_pitch): region minus discs; only materialised
                                 // for an external response map (eig_in), the fused path builds it per strip on chip
    int mask_pitch;
    float* eig;                  // unused by the fused path (kept for layout stability)
    const float* eig_in;         // nullable: externally supplied response map (seam op)
    unsigned long long* cand;    // candidate keys scratch [cand_cap]
    unsigned long long* cand2;   // second buffer [cand_cap]
    unsigned long long* cand3;   // third buffer [cand_cap]
    int cand_cap;
    int* cell_count;             // scratch [n_cells + 1]
    int* counters;               // [8]: 0 n_precand, 1 masked max (ordered int), 2 overflow flag (0..2 are reset by the selection
                                 //      kernel for the next launch), 3 n above threshold, 4 n_new, 5 M examined, 6 n_accepted,
                                 //      7 overflow flag of the last launch
    uint8_t* state;              // scratch [cand_cap]
    int* err;                    // nullable: sticky error word (bit 0: candidate buffer overflow)
    // point set the discs come from and new corners are appended to
    float2* pts;
    uint32_t* ids;               // nullable
    int32_t* track_cnt;          // nullable
    int* n;                      // current count (in/out)
    uint32_t* next_id;           // id counter (in/out), nullable
    int max_cnt;                 // capacity target: K = max_cnt - n
    int min_needed;              // detect only if K >= min_needed (1: TrackImage, 10: DetectNewFeature)
    int disc_radius;             // radius of the discs around existing points
    float min_dist;              // NMS distance
    double quality;              // 0.01
    int max_unmasked;            // 1: the quality threshold comes from the maximum over the WHOLE response map, not only the unmasked
                                 //    pixels (cv::cuda::GoodFeaturesToTrackDetector: cuda::minMax(eig) without the mask)
};
// marks (nullable): 3 events recorded after the mask fill, the discs and the response kernel;
// after_response (nullable): recorded between the response kernel and the (few-CTA) selection kernel
// level0_tmap (nullable): a CUtensorMap (128 bytes, dvfe_make_level0_tmap) over level 0 of the padded pyramids the jobs' images
// live in, job j at tensor row j * tma_rows_per_job: the response kernel then loads its tiles with TMA
int launch_gftt(const GfttJob* d_jobs, const GfttJob* h_jobs, int n_jobs, int max_w, int max_h, int max_pts,
                cudaStream_t st, cudaEvent_t* marks = nullptr, cudaEvent_t after_response = nullptr,
                const void* level0_tmap = nullptr, int tma_rows_per_job = 0);
// 2-D u8 tensor map over `n_rows` rows of `pitch` bytes at `base` with the response kernel's tile as box; out = 128 bytes.
// Returns DVFE_OK, or an error when the driver entry point is unavailable (the caller then launches without TMA).
int dvfe_make_level0_tmap(void* out, const uint8_t* base, int pitch, long n_rows);
int gftt_prepare_device();
int launch_min_eigen_val(const uint8_t* img, int pitch, int w, int h, float* eig, cudaStream_t st);
int launch_disc_mask(uint8_t* mask, int pitch, int w, int h, const float2* pts, const int* n, int max_pts, int radius,
                     cudaStream_t st);

// morph.cu
// label_mode: src is a label image (0 = background); the eroded image is inv_merge_mask = (label == 0 ? 255 : 0)
int launch_erode_rect(const uint8_t* src, int spitch, uint8_t* dst, int dpitch, uint8_t* tmp, int w, int h, int k,
                      int n_img, size_t img_stride, const int* enable, cudaStream_t st, int label_mode = 0);

int launch_erode_jobs(const ErodeJob* d_jobs, int n_jobs, int max_w, int max_h, cudaStream_t st);

// presence.cu: the extra work of a step in which some streams have no frame, no right image or start over
#define SF_TCACHE_VALID 0x80u    // stream flag byte, set by the host: the stream's forward-template cache matches its points
#define LANE_PRESENT 1u          // lane byte (d_lane): the stream has a frame in this step (0 = skipped)
#define LANE_STEREO 2u           // ... and a right image
struct PartialTables {
    const LkGroup* full_temporal;    // the tables of the step's buffer phase
    const LkGroup* full_stereo;
    const GfttJob* full_jobs;
    LkGroup* temporal;               // out
    LkGroup* stereo;                 // out
    GfttJob* jobs;                   // out
    uint8_t* lane;                   // out
    const int* zero;                 // a device 0: the point count of a stream a table leaves out
    int* n;                          // [B] point counts (RESET: 0)
    uint32_t* next_id;               // [B] id counters (RESET: 1)
};
int launch_partial_tables(const PartialTables& p, const uint8_t* d_sflags, int n_streams, int stereo_now, cudaStream_t st);
int launch_carry_pyramids(uint8_t* cur, const uint8_t* prev, size_t bytes, const uint8_t* d_sflags, int n_streams, cudaStream_t st);

// points.cu
struct CamParams {
    double inv_K11, inv_K13, inv_K22, inv_K23;
    double k1, k2, p1, p2;
    int no_distortion;
};
CamParams make_cam(const dvfe_camera& c);
int launch_lift(const CamParams& cam, const float2* pts, int n, float offx, float offy, float2* out, cudaStream_t st);
