// Upstream frame preparation (SURVEY.md §8f row N1) — the two byte-wise passes that bracket the hot path today:
//   SemanticImage::SetGrayImage[Gpu]   cv::cvtColor(color, gray, CV_BGR2GRAY)      basic/semantic_image.cpp:69-93
//   SemanticImage::SetMaskAndRoi / SetBackgroundMask: merge_mask = any(instance mask) * 255,
//                                       inv_merge_mask = bitwise_not(merge_mask)   basic/semantic_image.cpp:20-63,103-117
// Pure HBM-bandwidth kernels, 4 pixels per thread.  cvtColor arithmetic: the 15-bit fixed-point coefficients of the
// cv2 4.13 oracle, gray = (B*3735 + G*19235 + R*9798 + 16384) >> 15 (OpenCV 3.4's scalar path uses the 14-bit set
// 1868/9617/4899, which differs by one grey level on ~0.2 % of pixels; see DESIGN.md).
#include "kernels.cuh"

__global__ void __launch_bounds__(256) k_bgr_to_gray(const uint8_t* __restrict__ bgr, int spitch, uint8_t* __restrict__ gray,
                                                     int dpitch, int w, int h) {
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x0 >= w || y >= h) return;
    const uint8_t* s = bgr + (size_t)y * spitch + 3 * x0;
    uint8_t* d = gray + (size_t)y * dpitch + x0;
    unsigned out = 0;
    const int n = min(4, w - x0);
    if (n == 4 && ((uintptr_t)s & 3) == 0) {
        const unsigned* p = reinterpret_cast<const unsigned*>(s);        // 12 bytes: B G R B | G R B G | R B G R
        const unsigned w0 = __ldg(p), w1 = __ldg(p + 1), w2 = __ldg(p + 2);
        const unsigned px[4][3] = {{w0 & 255, (w0 >> 8) & 255, (w0 >> 16) & 255},
                                   {w0 >> 24, w1 & 255, (w1 >> 8) & 255},
                                   {(w1 >> 16) & 255, w1 >> 24, w2 & 255},
                                   {(w2 >> 8) & 255, (w2 >> 16) & 255, w2 >> 24}};
#pragma unroll
        for (int i = 0; i < 4; i++) out |= ((px[i][0] * 3735u + px[i][1] * 19235u + px[i][2] * 9798u + 16384u) >> 15) << (8 * i);
    } else {
        for (int i = 0; i < n; i++)
            out |= (((unsigned)s[3 * i] * 3735u + (unsigned)s[3 * i + 1] * 19235u + (unsigned)s[3 * i + 2] * 9798u + 16384u) >> 15) << (8 * i);
    }
    if (n == 4 && ((uintptr_t)d & 3) == 0) *reinterpret_cast<unsigned*>(d) = out;
    else for (int i = 0; i < n; i++) d[i] = (uint8_t)(out >> (8 * i));
}

__global__ void __launch_bounds__(256) k_merge_masks(const uint8_t* __restrict__ masks, int n_masks, size_t mask_stride,
                                                     int spitch, uint8_t* __restrict__ merge, uint8_t* __restrict__ inv,
                                                     int dpitch, int w, int h) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    unsigned any = 0;
    for (int i = 0; i < n_masks; i++) any |= masks[i * mask_stride + (size_t)y * spitch + x];
    const uint8_t m = any ? 255 : 0;
    merge[(size_t)y * dpitch + x] = m;
    inv[(size_t)y * dpitch + x] = (uint8_t)~m;
}

// ---- cv::remap (INTER_LINEAR, BORDER_CONSTANT 0) with fixed-point maps + BGR2GRAY: the frame ingest ------------------
// ImageProcessor::Run (image_process/image_process.cpp:105-126): un = cv::remap(color, left_undist_map1, left_undist_map2,
// INTER_LINEAR) with the CV_16SC2 / CV_16UC1 maps of cv::initUndistortRectifyMap (utils/camera_model.cpp:479-501), then
// cvtColor(BGR2GRAY).  OpenCV's fixed-point bilinear remap: (sx, sy) = map1, fx = map2 & 31, fy = (map2 >> 5) & 31, weights
// w = {(32-fx)(32-fy), fx(32-fy), (32-fx)fy, fx fy} * 32 (exact shorts, sum 2^15), taps outside the source = 0,
// dst = (sum w * tap + 2^14) >> 15 per channel == (sum (w/32) * tap + 512) >> 10.  One thread = 4 consecutive output
// pixels of up to INGEST_SPT streams: the map entries are loaded once and reused across streams (the maps are shared
// by all streams and stay in L2), the source taps are gathers served by L1/L2.  Streams with their own maps
// (dvfe_set_stream_undistort_maps) go through k_ingest_remap_each, which decodes each image's maps for that image.
#define INGEST_SPT 8

// taps of one output pixel whose 2 x 2 footprint is not fully inside the source (border pixels only)
template <int CH>
__device__ __noinline__ void remap_taps_border(const uint8_t* __restrict__ img, int pitch, int w, int h, int sx, int sy,
                                               int w00, int w01, int w10, int w11, unsigned out[CH]) {
    const bool x0 = (unsigned)sx < (unsigned)w, x1 = (unsigned)(sx + 1) < (unsigned)w;
    const bool y0 = (unsigned)sy < (unsigned)h, y1 = (unsigned)(sy + 1) < (unsigned)h;
    for (int c = 0; c < CH; c++) {
        int acc = 512;
        if (x0 && y0) acc += w00 * __ldg(img + (size_t)sy * pitch + sx * CH + c);
        if (x1 && y0) acc += w01 * __ldg(img + (size_t)sy * pitch + (sx + 1) * CH + c);
        if (x0 && y1) acc += w10 * __ldg(img + (size_t)(sy + 1) * pitch + sx * CH + c);
        if (x1 && y1) acc += w11 * __ldg(img + (size_t)(sy + 1) * pitch + (sx + 1) * CH + c);
        out[c] = (unsigned)acc >> 10;
    }
}

// d = a.s16[0] * b.u8[2h] + a.s16[1] * b.u8[2h+1] + c     (h = 0: lo, 1: hi)
__device__ __forceinline__ int prep_dp2a_lo(int a, unsigned b, int c) {
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ int prep_dp2a_hi(int a, unsigned b, int c) {
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// 6 consecutive bytes at p (any alignment) as two registers: lo = bytes 0..3, hi = bytes 4..7 (reads the 12 aligned bytes
// around them: the caller guarantees p + 12 stays inside the image)
__device__ __forceinline__ void prep_load6(const uint8_t* __restrict__ p, unsigned& lo, unsigned& hi) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const unsigned* wp = reinterpret_cast<const unsigned*>(a & ~(uintptr_t)3);
    const unsigned w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2);
    const int sh = (int)(a & 3) * 8;
    lo = __funnelshift_r(w0, w1, sh);
    hi = __funnelshift_r(w1, w2, sh);
}

// bilinear BGR sample from the two 6-byte rows (B G R B G R) of the 2 x 2 footprint: per channel the taps (top c, top 3+c,
// bottom c, bottom 3+c) are gathered into one register with PRMT and reduced with two dp2a against the packed weights
__device__ __forceinline__ void remap_bgr_words(const uint8_t* __restrict__ p, int pitch, int wa, int wb, unsigned out[3]) {
    unsigned tl, th, bl, bh;
    prep_load6(p, tl, th);
    prep_load6(p + pitch, bl, bh);
    const unsigned X0 = __byte_perm(tl, bl, 0x7430);        // t0 t3 b0 b3
    const unsigned H = __byte_perm(th, bh, 0x5410);         // t4 t5 b4 b5
    const unsigned U = __byte_perm(tl, bl, 0x6521);         // t1 t2 b1 b2
    const unsigned X1 = __byte_perm(U, H, 0x6240);          // t1 t4 b1 b4
    const unsigned X2 = __byte_perm(U, H, 0x7351);          // t2 t5 b2 b5
    out[0] = (unsigned)prep_dp2a_hi(wb, X0, prep_dp2a_lo(wa, X0, 512)) >> 10;
    out[1] = (unsigned)prep_dp2a_hi(wb, X1, prep_dp2a_lo(wa, X1, 512)) >> 10;
    out[2] = (unsigned)prep_dp2a_hi(wb, X2, prep_dp2a_lo(wa, X2, 512)) >> 10;
}

__device__ __forceinline__ unsigned gray_of(unsigned b, unsigned g, unsigned r) {
    return (b * 3735u + g * 19235u + r * 9798u + 16384u) >> 15;
}

// Unmapped images (gray copy / BGR -> gray): 4 consecutive output pixels x0.. of row y of image s (n of them inside the row),
// word loads, one 32-bit store.
template <int CH, bool KEEP>
__device__ __forceinline__ void ingest_rows_px(const IngestArgs& a, int s, int x0, int y, int n) {
    const uint8_t* __restrict__ row = a.src + (size_t)s * a.src_stride + (size_t)y * a.src_pitch + x0 * CH;
    uint8_t* d = a.dst + (size_t)s * a.dst_stride + (size_t)y * a.dst_pitch + x0 * (KEEP ? CH : 1);
    if (KEEP) {
        for (int i = 0; i < n * CH; i++) d[i] = __ldg(row + i);
        return;
    }
    unsigned packed = 0;
    if (n == 4 && ((uintptr_t)row & 3) == 0) {
        const unsigned* p = reinterpret_cast<const unsigned*>(row);
        if (CH == 3) {
            const unsigned w0 = __ldg(p), w1 = __ldg(p + 1), w2 = __ldg(p + 2);   // B G R B | G R B G | R B G R
            packed = gray_of(w0 & 255, (w0 >> 8) & 255, (w0 >> 16) & 255) |
                     gray_of(w0 >> 24, w1 & 255, (w1 >> 8) & 255) << 8 |
                     gray_of((w1 >> 16) & 255, w1 >> 24, w2 & 255) << 16 |
                     gray_of((w2 >> 8) & 255, (w2 >> 16) & 255, w2 >> 24) << 24;
        } else {
            packed = __ldg(p);
        }
    } else {
        for (int i = 0; i < n; i++)
            packed |= (CH == 3 ? gray_of(__ldg(row + 3 * i), __ldg(row + 3 * i + 1), __ldg(row + 3 * i + 2)) : __ldg(row + i)) << (8 * i);
    }
    if (n == 4 && ((uintptr_t)d & 3) == 0) *reinterpret_cast<unsigned*>(d) = packed;
    else for (int i = 0; i < n; i++) d[i] = (uint8_t)(packed >> (8 * i));
}

template <int CH, bool KEEP>
__global__ void __launch_bounds__(256) k_ingest_rows(IngestArgs a) {
    const int x0 = (blockIdx.x * 32 + threadIdx.x) * 4;
    const int y = blockIdx.y * 8 + threadIdx.y;
    if (x0 >= a.w || y >= a.h) return;
    const int n = min(4, a.w - x0);
    const int s_end = min(a.n_img, (int)(blockIdx.z + 1) * INGEST_SPT);
    for (int s = blockIdx.z * INGEST_SPT; s < s_end; s++) ingest_rows_px<CH, KEEP>(a, s, x0, y, n);
}

// The body of k_ingest_remap (below) for the maps (map1, map2) and the images [s_begin, s_end): the per-image kernel's remap.
// k_ingest_remap keeps its own copy of these lines: written as a call of this function it compiles to 4-11 more registers.
template <int CH, bool KEEP>
__device__ __forceinline__ void remap_images(const IngestArgs& a, const short* map1, const unsigned short* map2,
                                             int xb, int y, int s_begin, int s_end) {
    int off[4], wa[4], wb[4];          // byte offset of tap (0,0); weights packed w00 | w01 << 16, w10 | w11 << 16
    short sxs[4], sys[4];
    unsigned inside = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int x = xb + 32 * i;
        off[i] = 0; wa[i] = 0; wb[i] = 0; sxs[i] = 0; sys[i] = 0;
        if (x < a.w) {
            const size_t m = (size_t)y * a.w + x;
            const unsigned xy = __ldg(reinterpret_cast<const unsigned*>(map1) + m);
            const unsigned f = __ldg(map2 + m);
            const int sx = (short)(xy & 0xffff), sy = (short)(xy >> 16);
            const int fx = f & 31, fy = (f >> 5) & 31;
            sxs[i] = (short)sx; sys[i] = (short)sy;
            wa[i] = ((32 - fx) * (32 - fy)) | (fx * (32 - fy)) << 16;
            wb[i] = ((32 - fx) * fy) | (fx * fy) << 16;
            // inside = the 2 x 2 footprint is in the image AND (3 channels) the 12 aligned bytes the word path reads around
            // each 6-byte row stay inside the image buffer; everything else takes the bounds-checked path
            if ((unsigned)sx < (unsigned)(a.w - 1) && (unsigned)sy < (unsigned)(a.h - 1) &&
                (CH != 3 || (sy + 1) * a.src_pitch + sx * CH + 12 <= a.h * a.src_pitch)) {
                inside |= 1u << i;
                off[i] = sy * a.src_pitch + sx * CH;
            }
        }
    }
    for (int s = s_begin; s < s_end; s++) {
        const uint8_t* __restrict__ img = a.src + (size_t)s * a.src_stride;
        uint8_t* drow = a.dst + (size_t)s * a.dst_stride + (size_t)y * a.dst_pitch;
        unsigned res[4][CH];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            if (xb + 32 * i >= a.w) break;
            const int w00 = wa[i] & 0xffff, w01 = wa[i] >> 16, w10 = wb[i] & 0xffff, w11 = wb[i] >> 16;
            if (inside >> i & 1) {
                const uint8_t* p = img + off[i];
                if (CH == 3) {
                    remap_bgr_words(p, a.src_pitch, wa[i], wb[i], res[i]);
                } else {
#pragma unroll
                    for (int c = 0; c < CH; c++)
                        res[i][c] = (unsigned)(w00 * __ldg(p + c) + w01 * __ldg(p + CH + c) + w10 * __ldg(p + a.src_pitch + c) +
                                               w11 * __ldg(p + a.src_pitch + CH + c) + 512) >> 10;
                }
            } else {
                remap_taps_border<CH>(img, a.src_pitch, a.w, a.h, sxs[i], sys[i], w00, w01, w10, w11, res[i]);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int x = xb + 32 * i;
            if (x >= a.w) break;
            if (KEEP) {
#pragma unroll
                for (int c = 0; c < CH; c++) drow[x * CH + c] = (uint8_t)res[i][c];
            } else {
                drow[x] = (uint8_t)(CH == 3 ? gray_of(res[i][0], res[i][1], res[i][2]) : res[i][0]);
            }
        }
    }
}

// Remapped images: lane l owns the output pixels x = 128 * blockIdx.x + 32 * i + l (i < 4), so that each warp-wide
// gather touches the taps of 32 ADJACENT pixels (undistortion maps are smooth: one or two cache lines per load; with 4
// consecutive pixels per lane every load spans four lines and the kernel is bound by L1 wavefronts).  Everything that
// depends only on the maps (tap offset, the four weights, inside/outside) is decoded once and reused for the INGEST_SPT
// streams the thread loops over; all source reads are ld.global.nc, so the loads of the next stream are not ordered
// behind the stores of this one.
template <int CH, bool KEEP>
__global__ void __launch_bounds__(256) k_ingest_remap(IngestArgs a) {
    const int xb = blockIdx.x * 128 + threadIdx.x;
    const int y = blockIdx.y * 8 + threadIdx.y;
    if (xb >= a.w || y >= a.h) return;
    int off[4], wa[4], wb[4];          // byte offset of tap (0,0); weights packed w00 | w01 << 16, w10 | w11 << 16
    short sxs[4], sys[4];
    unsigned inside = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int x = xb + 32 * i;
        off[i] = 0; wa[i] = 0; wb[i] = 0; sxs[i] = 0; sys[i] = 0;
        if (x < a.w) {
            const size_t m = (size_t)y * a.w + x;
            const unsigned xy = __ldg(reinterpret_cast<const unsigned*>(a.map1) + m);
            const unsigned f = __ldg(a.map2 + m);
            const int sx = (short)(xy & 0xffff), sy = (short)(xy >> 16);
            const int fx = f & 31, fy = (f >> 5) & 31;
            sxs[i] = (short)sx; sys[i] = (short)sy;
            wa[i] = ((32 - fx) * (32 - fy)) | (fx * (32 - fy)) << 16;
            wb[i] = ((32 - fx) * fy) | (fx * fy) << 16;
            // inside = the 2 x 2 footprint is in the image AND (3 channels) the 12 aligned bytes the word path reads around
            // each 6-byte row stay inside the image buffer; everything else takes the bounds-checked path
            if ((unsigned)sx < (unsigned)(a.w - 1) && (unsigned)sy < (unsigned)(a.h - 1) &&
                (CH != 3 || (sy + 1) * a.src_pitch + sx * CH + 12 <= a.h * a.src_pitch)) {
                inside |= 1u << i;
                off[i] = sy * a.src_pitch + sx * CH;
            }
        }
    }
    const int s_end = min(a.n_img, (int)(blockIdx.z + 1) * INGEST_SPT);
    for (int s = blockIdx.z * INGEST_SPT; s < s_end; s++) {
        const uint8_t* __restrict__ img = a.src + (size_t)s * a.src_stride;
        uint8_t* drow = a.dst + (size_t)s * a.dst_stride + (size_t)y * a.dst_pitch;
        unsigned res[4][CH];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            if (xb + 32 * i >= a.w) break;
            const int w00 = wa[i] & 0xffff, w01 = wa[i] >> 16, w10 = wb[i] & 0xffff, w11 = wb[i] >> 16;
            if (inside >> i & 1) {
                const uint8_t* p = img + off[i];
                if (CH == 3) {
                    remap_bgr_words(p, a.src_pitch, wa[i], wb[i], res[i]);
                } else {
#pragma unroll
                    for (int c = 0; c < CH; c++)
                        res[i][c] = (unsigned)(w00 * __ldg(p + c) + w01 * __ldg(p + CH + c) + w10 * __ldg(p + a.src_pitch + c) +
                                               w11 * __ldg(p + a.src_pitch + CH + c) + 512) >> 10;
                }
            } else {
                remap_taps_border<CH>(img, a.src_pitch, a.w, a.h, sxs[i], sys[i], w00, w01, w10, w11, res[i]);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int x = xb + 32 * i;
            if (x >= a.w) break;
            if (KEEP) {
#pragma unroll
                for (int c = 0; c < CH; c++) drow[x * CH + c] = (uint8_t)res[i][c];
            } else {
                drow[x] = (uint8_t)(CH == 3 ? gray_of(res[i][0], res[i][1], res[i][2]) : res[i][0]);
            }
        }
    }
}

// Per-image maps (streams with their own undistortion maps): image blockIdx.z is remapped with maps[blockIdx.z], decoded for that
// image alone; an image without maps gets the pixels of k_ingest_rows.  The same tile of output pixels per block as the two
// kernels above, and the same arithmetic, so every image gets the bytes the shared-map kernel (or k_ingest_rows) writes for its maps.
template <int CH>
__global__ void __launch_bounds__(256) k_ingest_remap_each(IngestArgs a, const IngestMaps* __restrict__ maps) {
    const int s = blockIdx.z;
    const int y = blockIdx.y * 8 + threadIdx.y;
    const IngestMaps m = maps[s];
    if (m.map1 == nullptr) {
        const int x0 = (blockIdx.x * 32 + threadIdx.x) * 4;
        if (x0 >= a.w || y >= a.h) return;
        ingest_rows_px<CH, false>(a, s, x0, y, min(4, a.w - x0));
        return;
    }
    const int xb = blockIdx.x * 128 + threadIdx.x;
    if (xb >= a.w || y >= a.h) return;
    remap_images<CH, false>(a, m.map1, m.map2, xb, y, s, s + 1);
}

// Table form of the ingest (every stream's image in its own buffer, dvfe_track_frames): image blockIdx.z is read through its table
// entry, at its own pitch, and gets the bytes k_ingest_remap_each writes (k_ingest_remap / k_ingest_rows with shared maps)
template <int CH>
__global__ void __launch_bounds__(256) k_ingest_table(IngestArgs a, const ImgSrc* __restrict__ srcs, const IngestMaps* __restrict__ maps) {
    const int s = blockIdx.z;
    const ImgSrc src = srcs[s];
    if (src.ptr == nullptr) return;
    a.src = src.ptr; a.src_pitch = src.pitch;
    a.dst += (size_t)s * a.dst_stride;
    const IngestMaps m = maps ? maps[s] : IngestMaps{a.map1, a.map2};
    const int y = blockIdx.y * 8 + threadIdx.y;
    if (m.map1 == nullptr) {
        const int x0 = (blockIdx.x * 32 + threadIdx.x) * 4;
        if (x0 >= a.w || y >= a.h) return;
        ingest_rows_px<CH, false>(a, 0, x0, y, min(4, a.w - x0));
        return;
    }
    const int xb = blockIdx.x * 128 + threadIdx.x;
    if (xb >= a.w || y >= a.h) return;
    remap_images<CH, false>(a, m.map1, m.map2, xb, y, 0, 1);
}

int launch_ingest_table(const IngestArgs& a, const ImgSrc* d_src, cudaStream_t st, const IngestMaps* d_maps) {
    if (a.n_img <= 0) return DVFE_OK;
    if (a.keep_channels) { dvfe_set_error("ingest: the table form writes gray images only"); return DVFE_ERR_INVALID; }
    const dim3 blk(32, 8), grid((a.w + 127) / 128, (a.h + 7) / 8, a.n_img);
    if (a.ch == 3) DVFE_LAUNCH((k_ingest_table<3>), grid, blk, 0, st, a, d_src, d_maps);
    else DVFE_LAUNCH((k_ingest_table<1>), grid, blk, 0, st, a, d_src, d_maps);
    return DVFE_OK;
}

// image blockIdx.z of the table, 4 bytes per thread (word copies where both sides are aligned)
__global__ void __launch_bounds__(256) k_gather_images(const ImgSrc* __restrict__ srcs, uint8_t* __restrict__ dst, size_t dst_stride,
                                                       int dst_pitch, int row, int h) {
    const ImgSrc src = srcs[blockIdx.z];
    if (src.ptr == nullptr) return;
    const int x0 = (blockIdx.x * 32 + threadIdx.x) * 4, y = blockIdx.y * 8 + threadIdx.y;
    if (x0 >= row || y >= h) return;
    const uint8_t* s = src.ptr + (size_t)y * src.pitch + x0;
    uint8_t* d = dst + (size_t)blockIdx.z * dst_stride + (size_t)y * dst_pitch + x0;
    const int n = min(4, row - x0);
    if (n == 4 && (((uintptr_t)s | (uintptr_t)d) & 3) == 0) *reinterpret_cast<unsigned*>(d) = __ldg(reinterpret_cast<const unsigned*>(s));
    else for (int i = 0; i < n; i++) d[i] = __ldg(s + i);
}

int launch_gather_images(const ImgSrc* d_src, uint8_t* dst, size_t dst_stride, int dst_pitch, int row, int h, int n_img,
                         cudaStream_t st) {
    if (n_img <= 0) return DVFE_OK;
    const dim3 blk(32, 8), grid(((row + 3) / 4 + 31) / 32, (h + 7) / 8, n_img);
    DVFE_LAUNCH(k_gather_images, grid, blk, 0, st, d_src, dst, dst_stride, dst_pitch, row, h);
    return DVFE_OK;
}

int launch_ingest(const IngestArgs& a, cudaStream_t st, const IngestMaps* d_maps) {
    if (a.n_img <= 0) return DVFE_OK;
    const int nz = (a.n_img + INGEST_SPT - 1) / INGEST_SPT;
    dim3 blk(32, 8), grid((a.w + 127) / 128, (a.h + 7) / 8, nz);
    if (d_maps) {
        if (a.keep_channels) { dvfe_set_error("ingest: per-image maps write gray images only"); return DVFE_ERR_INVALID; }
        const dim3 grid_each(grid.x, grid.y, a.n_img);
        if (a.ch == 3) DVFE_LAUNCH((k_ingest_remap_each<3>), grid_each, blk, 0, st, a, d_maps);
        else DVFE_LAUNCH((k_ingest_remap_each<1>), grid_each, blk, 0, st, a, d_maps);
    } else if (a.map1) {
        if (a.ch == 3 && a.keep_channels) DVFE_LAUNCH((k_ingest_remap<3, true>), grid, blk, 0, st, a);
        else if (a.ch == 3) DVFE_LAUNCH((k_ingest_remap<3, false>), grid, blk, 0, st, a);
        else DVFE_LAUNCH((k_ingest_remap<1, false>), grid, blk, 0, st, a);
    } else {
        if (a.ch == 3 && a.keep_channels) DVFE_LAUNCH((k_ingest_rows<3, true>), grid, blk, 0, st, a);
        else if (a.ch == 3) DVFE_LAUNCH((k_ingest_rows<3, false>), grid, blk, 0, st, a);
        else DVFE_LAUNCH((k_ingest_rows<1, false>), grid, blk, 0, st, a);
    }
    return DVFE_OK;
}

extern "C" int dvfe_op_remap(const uint8_t* src, int w, int h, int channels, int pitch, const int16_t* map1,
                             const uint16_t* map2, int to_gray, uint8_t* dst) {
    if (!src || !dst || w < 1 || h < 1 || (channels != 1 && channels != 3) || pitch < channels * w || (map1 != nullptr) != (map2 != nullptr)) {
        dvfe_set_error("op_remap: bad argument");
        return DVFE_ERR_INVALID;
    }
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) { dvfe_set_error("no CUDA device available: libdvfe has no CPU fallback"); return DVFE_ERR_NO_DEVICE; }
    const size_t P = (size_t)w * h;
    const int och = (channels == 3 && !to_gray) ? 3 : 1;
    uint8_t *d_src = nullptr, *d_dst = nullptr;
    short* d_m1 = nullptr;
    unsigned short* d_m2 = nullptr;
    cudaError_t e = cudaMalloc((void**)&d_src, P * channels);
    if (e == cudaSuccess) e = cudaMalloc((void**)&d_dst, P * och);
    if (e == cudaSuccess && map1) e = cudaMalloc((void**)&d_m1, P * 4);
    if (e == cudaSuccess && map1) e = cudaMalloc((void**)&d_m2, P * 2);
    if (e == cudaSuccess) e = cudaMemcpy2D(d_src, (size_t)channels * w, src, pitch, (size_t)channels * w, h, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && map1) e = cudaMemcpy(d_m1, map1, P * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && map1) e = cudaMemcpy(d_m2, map2, P * 2, cudaMemcpyHostToDevice);
    int rc = DVFE_OK;
    if (e == cudaSuccess) {
        IngestArgs a{d_src, P * channels, channels * w, channels, d_m1, d_m2, d_dst, P * och, och * w, w, h, 1, och == 3 ? 1 : 0};
        rc = launch_ingest(a, 0);
        if (rc == DVFE_OK) e = cudaDeviceSynchronize();
        if (rc == DVFE_OK && e == cudaSuccess) e = cudaMemcpy(dst, d_dst, P * och, cudaMemcpyDeviceToHost);
    }
    cudaFree(d_src); cudaFree(d_dst); cudaFree(d_m1); cudaFree(d_m2);
    if (rc != DVFE_OK) return rc;
    if (e != cudaSuccess) { dvfe_set_error("op_remap: %s", cudaGetErrorString(e)); return DVFE_ERR_CUDA; }
    return DVFE_OK;
}

namespace {
struct PrepBuf {                 // device buffer freed on every exit path
    void* p = nullptr;
    ~PrepBuf() { if (p) cudaFree(p); }
    int alloc(size_t bytes) {
        DVFE_CUDA(cudaMalloc(&p, bytes ? bytes : 1));
        return DVFE_OK;
    }
    template <typename T> T* as() { return reinterpret_cast<T*>(p); }
};
int prep_device() {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
        dvfe_set_error("no CUDA device available: libdvfe has no CPU fallback");
        return DVFE_ERR_NO_DEVICE;
    }
    return DVFE_OK;
}
}  // namespace

extern "C" int dvfe_op_bgr_to_gray(const uint8_t* bgr, int w, int h, int pitch, uint8_t* gray_out) {
    if (!bgr || !gray_out || w < 1 || h < 1 || pitch < 3 * w) { dvfe_set_error("op_bgr_to_gray: bad argument"); return DVFE_ERR_INVALID; }
    if (int rc = prep_device()) return rc;
    PrepBuf d_bgr, d_gray;
    if (int rc = d_bgr.alloc((size_t)3 * w * h)) return rc;
    if (int rc = d_gray.alloc((size_t)w * h)) return rc;
    DVFE_CUDA(cudaMemcpy2D(d_bgr.p, (size_t)3 * w, bgr, pitch, (size_t)3 * w, h, cudaMemcpyHostToDevice));
    dim3 blk(32, 8), grid(((w + 3) / 4 + 31) / 32, (h + 7) / 8);
    DVFE_LAUNCH(k_bgr_to_gray, grid, blk, 0, 0, d_bgr.as<uint8_t>(), 3 * w, d_gray.as<uint8_t>(), w, w, h);
    DVFE_CUDA(cudaDeviceSynchronize());
    DVFE_CUDA(cudaMemcpy(gray_out, d_gray.p, (size_t)w * h, cudaMemcpyDeviceToHost));
    return DVFE_OK;
}

extern "C" int dvfe_op_merge_masks(const uint8_t* masks, int n_masks, int w, int h, uint8_t* merge_out, uint8_t* inv_out) {
    if (n_masks < 0 || (n_masks > 0 && !masks) || !merge_out || !inv_out || w < 1 || h < 1) {
        dvfe_set_error("op_merge_masks: bad argument");
        return DVFE_ERR_INVALID;
    }
    if (int rc = prep_device()) return rc;
    const size_t P = (size_t)w * h;
    PrepBuf d_m, d_merge, d_inv;
    if (int rc = d_m.alloc(P * (n_masks > 0 ? n_masks : 1))) return rc;
    if (int rc = d_merge.alloc(P)) return rc;
    if (int rc = d_inv.alloc(P)) return rc;
    if (n_masks > 0) DVFE_CUDA(cudaMemcpy(d_m.p, masks, P * n_masks, cudaMemcpyHostToDevice));
    dim3 blk(32, 8), grid((w + 31) / 32, (h + 7) / 8);
    DVFE_LAUNCH(k_merge_masks, grid, blk, 0, 0, d_m.as<uint8_t>(), n_masks, P, w, d_merge.as<uint8_t>(), d_inv.as<uint8_t>(), w, w, h);
    DVFE_CUDA(cudaDeviceSynchronize());
    DVFE_CUDA(cudaMemcpy(merge_out, d_merge.p, P, cudaMemcpyDeviceToHost));
    DVFE_CUDA(cudaMemcpy(inv_out, d_inv.p, P, cudaMemcpyDeviceToHost));
    return DVFE_OK;
}

// FeatureTrack(): "remove the masks of static objects" (system/main.cpp:219-242): for every pixel of a static instance's
// ROI mask that is set, merge_mask = 0; afterwards inv_merge_mask = bitwise_not(merge_mask) (:238-240).
__global__ void __launch_bounds__(256) k_punch_out(uint8_t* __restrict__ merge, uint8_t* __restrict__ inv, int pitch, int w, int h,
                                                   const uint8_t* __restrict__ roi, int roi_pitch, int rx, int ry, int rw, int rh) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= rw || y >= rh) return;
    const int gx = rx + x, gy = ry + y;
    if (gx < 0 || gx >= w || gy < 0 || gy >= h) return;
    if (roi[(size_t)y * roi_pitch + x] != 0) {           // mask_cv.at<uchar>(row, col) >= 0.5
        merge[(size_t)gy * pitch + gx] = 0;
        inv[(size_t)gy * pitch + gx] = 255;
    }
}

extern "C" int dvfe_op_punch_out(uint8_t* merge_mask, uint8_t* inv_merge_mask, int w, int h, const uint8_t* roi_mask,
                                 int roi_pitch, int x, int y, int roi_w, int roi_h) {
    if (!merge_mask || !inv_merge_mask || !roi_mask || w < 1 || h < 1 || roi_w < 1 || roi_h < 1 || roi_pitch < roi_w) {
        dvfe_set_error("op_punch_out: bad argument");
        return DVFE_ERR_INVALID;
    }
    if (int rc = prep_device()) return rc;
    const size_t P = (size_t)w * h;
    PrepBuf d_merge, d_inv, d_roi;
    if (int rc = d_merge.alloc(P)) return rc;
    if (int rc = d_inv.alloc(P)) return rc;
    if (int rc = d_roi.alloc((size_t)roi_w * roi_h)) return rc;
    DVFE_CUDA(cudaMemcpy(d_merge.p, merge_mask, P, cudaMemcpyHostToDevice));
    DVFE_CUDA(cudaMemcpy(d_inv.p, inv_merge_mask, P, cudaMemcpyHostToDevice));
    DVFE_CUDA(cudaMemcpy2D(d_roi.p, roi_w, roi_mask, roi_pitch, roi_w, roi_h, cudaMemcpyHostToDevice));
    dim3 blk(32, 8), grid((roi_w + 31) / 32, (roi_h + 7) / 8);
    DVFE_LAUNCH(k_punch_out, grid, blk, 0, 0, d_merge.as<uint8_t>(), d_inv.as<uint8_t>(), w, w, h, d_roi.as<uint8_t>(), roi_w, x, y,
                roi_w, roi_h);
    DVFE_CUDA(cudaDeviceSynchronize());
    DVFE_CUDA(cudaMemcpy(merge_mask, d_merge.p, P, cudaMemcpyDeviceToHost));
    DVFE_CUDA(cudaMemcpy(inv_merge_mask, d_inv.p, P, cudaMemcpyDeviceToHost));
    return DVFE_OK;
}
