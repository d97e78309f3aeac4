// Image pyramid build — replaces cv::buildOpticalFlowPyramid as called inside
// cv::calcOpticalFlowPyrLK (reference call sites: dynamic_vins/src/front_end/feature_utils.cpp:43,50).
//   level 0 = the image; level l = pyrDown(level l-1): separable [1 4 6 4 1], BORDER_REFLECT_101,
//   (sum + 128) >> 8, size ((w+1)/2, (h+1)/2).  Integer arithmetic, bit-exact.
// Every level is written once, with a REFLECT_101 border (common.cuh), and is then reused by the
// temporal LK of this frame, the stereo LK of this frame and the temporal LK of the next frame
// (the reference rebuilds both pyramids inside each of its 4 LK calls per stereo frame).
#include <stdlib.h>

#include "kernels.cuh"

__device__ __forceinline__ void pyr_select(const PyrImgSet& set, int img, const uint8_t*& src, uint8_t*& dst) {
    const bool second = img >= set.per_set;
    const int idx = second ? img - set.per_set : img;
    src = (second ? set.src[1] : set.src[0]) + (size_t)idx * set.src_stride;
    dst = (second ? set.dst[1] : set.dst[0]) + (size_t)idx * set.dst_stride;
}

// ---- level 0: copy the u8 image into the padded level; one thread = 16 bytes ------------------
// fuse_border (pyr_level0_fusable: w and padR multiples of 16, single reflections, the right-edge threads not lane 0 of their
// warp): the thread also stores the REFLECT_101 border words its pixels mirror into (byte permutations of adjacent words, the
// neighbour's word by warp shuffle) and the rows above / below the image that mirror its row: no border launch for level 0.
__host__ __device__ __forceinline__ bool pyr_level0_fusable(const PyrLevel& L) {
    const int padR = L.pitch - DVFE_PADX - L.w;
    if ((L.w & 15) != 0 || (padR & 15) != 0 || L.w <= DVFE_PADX + 16 || L.w <= padR + 16 || L.h <= DVFE_PADY + 1) return false;
    for (int q = 0; q * 16 < padR; q++)
        if (((L.w / 16 - 1 - q) & 31) == 0) return false;
    return true;
}

__global__ void __launch_bounds__(256) k_pyr_level0(PyrImgSet set, PyrLevel L, int spitch, int fuse_border) {
    const uint8_t* src; uint8_t* dst;
    pyr_select(set, blockIdx.z, src, dst);
    dst += L.offset + (size_t)DVFE_PADY * L.pitch + DVFE_PADX;
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x0 >= L.w || y >= L.h) return;
    const uint8_t* row = src + (size_t)y * spitch + x0;
    uint8_t* out = dst + (size_t)y * L.pitch + x0;
    uint4 q;
    if (x0 + 15 < L.w && (((uintptr_t)row) & 15) == 0) {
        q = __ldg(reinterpret_cast<const uint4*>(row));
    } else if (x0 + 15 < L.w && (((uintptr_t)row) & 3) == 0) {
        const unsigned* p = reinterpret_cast<const unsigned*>(row);
        q = make_uint4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
    } else if (x0 + 15 < L.w) {
        unsigned w4[4];
#pragma unroll
        for (int i = 0; i < 4; i++)
            w4[i] = (unsigned)__ldg(row + 4 * i) | ((unsigned)__ldg(row + 4 * i + 1) << 8) | ((unsigned)__ldg(row + 4 * i + 2) << 16) |
                    ((unsigned)__ldg(row + 4 * i + 3) << 24);
        q = make_uint4(w4[0], w4[1], w4[2], w4[3]);
    } else {
        for (int i = 0; i < 16 && x0 + i < L.w; i++) out[i] = __ldg(row + i);      // ragged last column (never with fuse_border)
        return;
    }
    *reinterpret_cast<uint4*>(out) = q;
    if (!fuse_border) return;
    const unsigned am = __activemask();
    const unsigned nxt = __shfl_down_sync(am, q.x, 1), prv = __shfl_up_sync(am, q.w, 1);
    const int padR = L.pitch - DVFE_PADX - L.w, q16 = L.w - 16 - x0;
    const bool left = x0 < DVFE_PADX, right = q16 < padR;
    int ys[3], ny = 1;
    ys[0] = y;
    if (y >= 1 && y <= DVFE_PADY) ys[ny++] = -y;
    if (y <= L.h - 2 && y >= L.h - 1 - DVFE_PADY) ys[ny++] = 2 * (L.h - 1) - y;
    if (!left && !right && ny == 1) return;
    // pixels x0+1 .. x0+16 reversed -> x' = -x0-16 .. -x0-1 ; pixels x0-1 .. x0+14 reversed -> x' = w+q16 .. w+q16+15
    const uint4 lb = make_uint4(__byte_perm(q.w, nxt, 0x1234), __byte_perm(q.z, q.w, 0x1234), __byte_perm(q.y, q.z, 0x1234),
                                __byte_perm(q.x, q.y, 0x1234));
    const uint4 rb = make_uint4(__byte_perm(q.w, q.z, 0x7012), __byte_perm(q.z, q.y, 0x7012), __byte_perm(q.y, q.x, 0x7012),
                                __byte_perm(q.x, prv, 0x7012));
    for (int j = 0; j < ny; j++) {
        uint8_t* __restrict__ orow = dst + (ptrdiff_t)ys[j] * L.pitch;
        if (j > 0) *reinterpret_cast<uint4*>(orow + x0) = q;
        if (left) *reinterpret_cast<uint4*>(orow - x0 - 16) = lb;
        if (right) *reinterpret_cast<uint4*>(orow + L.w + q16) = rb;
    }
}

// The body of k_pyr_level0 for one image (dst = pixel (0,0) of the level), for the table form below.  k_pyr_level0 keeps its own
// copy of these lines: written as a call of this function it compiles to another register count.
__device__ __forceinline__ void pyr_level0_body(const uint8_t* src, uint8_t* dst, const PyrLevel& L, int spitch, int fuse_border) {
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x0 >= L.w || y >= L.h) return;
    const uint8_t* row = src + (size_t)y * spitch + x0;
    uint8_t* out = dst + (size_t)y * L.pitch + x0;
    uint4 q;
    if (x0 + 15 < L.w && (((uintptr_t)row) & 15) == 0) {
        q = __ldg(reinterpret_cast<const uint4*>(row));
    } else if (x0 + 15 < L.w && (((uintptr_t)row) & 3) == 0) {
        const unsigned* p = reinterpret_cast<const unsigned*>(row);
        q = make_uint4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
    } else if (x0 + 15 < L.w) {
        unsigned w4[4];
#pragma unroll
        for (int i = 0; i < 4; i++)
            w4[i] = (unsigned)__ldg(row + 4 * i) | ((unsigned)__ldg(row + 4 * i + 1) << 8) | ((unsigned)__ldg(row + 4 * i + 2) << 16) |
                    ((unsigned)__ldg(row + 4 * i + 3) << 24);
        q = make_uint4(w4[0], w4[1], w4[2], w4[3]);
    } else {
        for (int i = 0; i < 16 && x0 + i < L.w; i++) out[i] = __ldg(row + i);      // ragged last column (never with fuse_border)
        return;
    }
    *reinterpret_cast<uint4*>(out) = q;
    if (!fuse_border) return;
    const unsigned am = __activemask();
    const unsigned nxt = __shfl_down_sync(am, q.x, 1), prv = __shfl_up_sync(am, q.w, 1);
    const int padR = L.pitch - DVFE_PADX - L.w, q16 = L.w - 16 - x0;
    const bool left = x0 < DVFE_PADX, right = q16 < padR;
    int ys[3], ny = 1;
    ys[0] = y;
    if (y >= 1 && y <= DVFE_PADY) ys[ny++] = -y;
    if (y <= L.h - 2 && y >= L.h - 1 - DVFE_PADY) ys[ny++] = 2 * (L.h - 1) - y;
    if (!left && !right && ny == 1) return;
    // pixels x0+1 .. x0+16 reversed -> x' = -x0-16 .. -x0-1 ; pixels x0-1 .. x0+14 reversed -> x' = w+q16 .. w+q16+15
    const uint4 lb = make_uint4(__byte_perm(q.w, nxt, 0x1234), __byte_perm(q.z, q.w, 0x1234), __byte_perm(q.y, q.z, 0x1234),
                                __byte_perm(q.x, q.y, 0x1234));
    const uint4 rb = make_uint4(__byte_perm(q.w, q.z, 0x7012), __byte_perm(q.z, q.y, 0x7012), __byte_perm(q.y, q.x, 0x7012),
                                __byte_perm(q.x, prv, 0x7012));
    for (int j = 0; j < ny; j++) {
        uint8_t* __restrict__ orow = dst + (ptrdiff_t)ys[j] * L.pitch;
        if (j > 0) *reinterpret_cast<uint4*>(orow + x0) = q;
        if (left) *reinterpret_cast<uint4*>(orow - x0 - 16) = lb;
        if (right) *reinterpret_cast<uint4*>(orow + L.w + q16) = rb;
    }
}

// one image per grid z, read through the stream's table entry; the whole block leaves when the image is absent
__global__ void __launch_bounds__(256) k_pyr_level0_table(const ImgSrc* __restrict__ srcs, uint8_t* dst, size_t dst_stride,
                                                          PyrLevel L, int fuse_border) {
    const ImgSrc src = srcs[blockIdx.z];
    if (src.ptr == nullptr) return;
    pyr_level0_body(src.ptr, dst + (size_t)blockIdx.z * dst_stride + L.offset + (size_t)DVFE_PADY * L.pitch + DVFE_PADX, L,
                    src.pitch, fuse_border);
}

// ---- REFLECT_101 border of a level, copied from its own interior; one warp per padded row ------------------
// Word path (w a multiple of 4, single reflections): an interior word of a band row is an aligned copy; a left border word is
// the byte permutation (W[j+1].b0, W[j].b3, W[j].b2, W[j].b1) of two adjacent interior words of the source row, a right border
// word (V[m].b2, V[m].b1, V[m].b0, V[m+1].b3) with V[t] = the t-th word from the right end.  Other shapes: byte by byte.
__device__ __forceinline__ void pyr_border_body(uint8_t* base, const PyrLevel& L, int py, int lane) {
    uint8_t* lvl = base + L.offset;
    const uint8_t* __restrict__ in = lvl + (size_t)DVFE_PADY * L.pitch + DVFE_PADX;      // pixel (0,0)
    if (py >= L.h + 2 * DVFE_PADY) return;
    const int y = py - DVFE_PADY;
    const uint8_t* __restrict__ srow = in + (size_t)reflect101(y, L.h) * L.pitch;
    unsigned* orow = reinterpret_cast<unsigned*>(lvl + (size_t)py * L.pitch);
    const int nwords = L.pitch / 4;
    const int right0 = (DVFE_PADX + L.w) / 4;          // first word that holds a right-border byte
    const bool band = y < 0 || y >= L.h;
    // band rows: every word; side rows: the left pad words, then the words from right0 on
    const int count = band ? nwords : (DVFE_PADX / 4 + nwords - right0);
    const int padR = L.pitch - DVFE_PADX - L.w;
    if ((L.w & 3) == 0 && L.w > DVFE_PADX + 4 && L.w > padR + 4) {
        const unsigned* __restrict__ sw = reinterpret_cast<const unsigned*>(srow);       // interior words of the source row
        const int iw = L.w / 4;
        for (int t = lane; t < count; t += 32) {
            const int wq = band ? t : (t < DVFE_PADX / 4 ? t : right0 + (t - DVFE_PADX / 4));
            const int k = wq - DVFE_PADX / 4;          // interior word index (negative: left border, >= iw: right border)
            unsigned v;
            if (k < 0) { const int j = -k - 1; v = __byte_perm(sw[j], sw[j + 1], 0x1234); }
            else if (k >= iw) { const int m = k - iw; v = __byte_perm(sw[iw - 1 - m], sw[iw - 2 - m], 0x7012); }
            else v = sw[k];
            orow[wq] = v;
        }
        return;
    }
    for (int t = lane; t < count; t += 32) {
        const int wq = band ? t : (t < DVFE_PADX / 4 ? t : right0 + (t - DVFE_PADX / 4));
        const int x0 = wq * 4 - DVFE_PADX;
        unsigned v = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) v |= (unsigned)srow[reflect101(x0 + i, L.w)] << (8 * i);
        orow[wq] = v;
    }
}

// Word-path border of one level with every thread busy: a block takes 256 border words.  Blocks [0, side_blocks) cover the side
// rows (rows_per_block rows x (PADX/4 + padR/4) words each), the blocks after them the 2 * PADY band rows (all pitch/4 words).
__host__ __device__ __forceinline__ bool pyr_border_words_ok(const PyrLevel& L) {
    const int padR = L.pitch - DVFE_PADX - L.w;
    return (L.w & 3) == 0 && L.w > DVFE_PADX + 4 && L.w > padR + 4 && L.h > DVFE_PADY;
}

__global__ void __launch_bounds__(256) k_pyr_border_words(PyrImgSet set, PyrLevel L, int side_blocks) {
    const uint8_t* src; uint8_t* base;
    pyr_select(set, blockIdx.z, src, base);
    uint8_t* lvl = base + L.offset;
    const int nwords = L.pitch / 4, iw = L.w / 4, lw = DVFE_PADX / 4;
    const int swn = nwords - iw;                       // border words of a side row: lw on the left, the rest on the right
    int py, wq;
    if ((int)blockIdx.x < side_blocks) {
        const int rpb = 256 / swn;
        const int r = threadIdx.x / swn, t = threadIdx.x - r * swn;
        const int y = blockIdx.x * rpb + r;
        if (r >= rpb || y >= L.h) return;
        py = y + DVFE_PADY;
        wq = t < lw ? t : iw + t;                      // right border words start at lw + iw
    } else {
        const int t = (blockIdx.x - side_blocks) * 256 + threadIdx.x;
        const int r = t / nwords;
        if (r >= 2 * DVFE_PADY) return;
        wq = t - r * nwords;
        py = r < DVFE_PADY ? r : L.h + r;              // rows above, then rows below the image
    }
    const int y = py - DVFE_PADY;
    const int ys = y < 0 ? -y : (y >= L.h ? 2 * (L.h - 1) - y : y);          // single reflection (h > PADY)
    const unsigned* __restrict__ sw = reinterpret_cast<const unsigned*>(lvl + (size_t)(ys + DVFE_PADY) * L.pitch + DVFE_PADX);
    const int k = wq - lw;
    unsigned v;
    if (k < 0) { const int j = -k - 1; v = __byte_perm(sw[j], sw[j + 1], 0x1234); }
    else if (k >= iw) { const int m = k - iw; v = __byte_perm(sw[iw - 1 - m], sw[iw - 2 - m], 0x7012); }
    else v = sw[k];
    reinterpret_cast<unsigned*>(lvl + (size_t)py * L.pitch)[wq] = v;
}

__global__ void k_pyr_border(PyrImgSet set, PyrLevel L);

static int launch_pyr_border(const PyrImgSet& set, int n_img, const PyrLevel& D, cudaStream_t st) {
    if (pyr_border_words_ok(D)) {
        const int nwords = D.pitch / 4, swn = nwords - D.w / 4, rpb = 256 / swn;
        const int side_blocks = (D.h + rpb - 1) / rpb, band_blocks = (2 * DVFE_PADY * nwords + 255) / 256;
        DVFE_LAUNCH(k_pyr_border_words, dim3(side_blocks + band_blocks, 1, n_img), 256, 0, st, set, D, side_blocks);
    } else {
        dim3 bgrid((D.h + 2 * DVFE_PADY + 7) / 8, 1, n_img);
        DVFE_LAUNCH(k_pyr_border, bgrid, dim3(32, 8), 0, st, set, D);
    }
    return DVFE_OK;
}

__global__ void __launch_bounds__(256) k_pyr_border(PyrImgSet set, PyrLevel L) {
    const uint8_t* src; uint8_t* base;
    pyr_select(set, blockIdx.z, src, base);
    pyr_border_body(base, L, blockIdx.x * blockDim.y + threadIdx.y, threadIdx.x);
}

__global__ void __launch_bounds__(256) k_pyr_border_jobs(const PyrJob* __restrict__ jobs, int level) {
    const PyrJob& J = jobs[blockIdx.z];
    if (level >= J.desc.n_levels) return;
    pyr_border_body(J.dst, J.desc.lv[level], blockIdx.x * blockDim.y + threadIdx.y, threadIdx.x);
}

// ---- level l interior from level l-1 (padded, border already filled) -------------------------------------
__device__ __forceinline__ int pyr_tap5(const uint8_t* __restrict__ p) {
    return (int)p[-2] + 4 * (int)p[-1] + 6 * (int)p[0] + 4 * (int)p[1] + (int)p[2];
}

// ---- REFLECT_101 border written by the threads that produce the interior (levels >= 1 of the batched pyramids) ----
// Border position x' = -d (1 <= d <= PADX) holds pixel d, x' = w-1+d (1 <= d <= padR, padR = pitch - PADX - w) holds pixel
// w-1-d; rows likewise with PADY above and below.  When every border position is the single reflection of an interior pixel,
// the thread that computes a pixel can store its mirror images itself and the separate k_pyr_border launch of that level
// disappears.  Done with whole words: a thread holds 8 pixels = 2 words of a row; a border word is a byte permutation of two
// adjacent row words (__byte_perm), the second of which comes from the neighbouring thread by warp shuffle.  Conditions
// (pyr_border_fusable): w a multiple of 8 (no ragged thread column; padR is then a multiple of 8 too), w > PADX + 8 and
// w > padR + 8 (single reflection, neighbour exists), h > PADY + 1, and no right-edge thread is lane 0 of its warp.
__host__ __device__ __forceinline__ bool pyr_border_fusable(const PyrLevel& L) {
    const int padR = L.pitch - DVFE_PADX - L.w;
    if ((L.w & 7) != 0 || L.w <= DVFE_PADX + 8 || L.w <= padR + 8 || L.h <= DVFE_PADY + 1) return false;
    for (int q = 0; q * 8 < padR; q++)
        if (((L.w / 8 - 1 - q) & 31) == 0) return false;
    return true;
}

// one pixel and its mirror images (ragged bottom row of the interior: odd h)
__device__ __forceinline__ void pyr_store_px_mirrored(uint8_t* __restrict__ dst, const PyrLevel& D, int x, int y, uint8_t v) {
    const int padR = D.pitch - DVFE_PADX - D.w;
    int xs[3], ys[3], nx = 1, ny = 1;
    xs[0] = x; ys[0] = y;
    if (x >= 1 && x <= DVFE_PADX) xs[nx++] = -x;
    if (x <= D.w - 2 && x >= D.w - 1 - padR) xs[nx++] = 2 * (D.w - 1) - x;
    if (y >= 1 && y <= DVFE_PADY) ys[ny++] = -y;
    if (y <= D.h - 2 && y >= D.h - 1 - DVFE_PADY) ys[ny++] = 2 * (D.h - 1) - y;
    for (int j = 0; j < ny; j++)
        for (int i = 0; i < nx; i++) dst[(ptrdiff_t)ys[j] * D.pitch + xs[i]] = v;
}

// Row y of the fused fast path: v = pixels x0..x0+7, nxt = first word of the next thread's pixels, prv = last word of the
// previous thread's.  Stores the interior words and, for edge threads, the border words they mirror into; the same for the
// rows above / below the image that mirror row y.
__device__ __forceinline__ void pyr_store8_fused(uint8_t* __restrict__ dst, const PyrLevel& D, int x0, int y, uint2 v, unsigned nxt,
                                                 unsigned prv) {
    const int padR = D.pitch - DVFE_PADX - D.w;
    const bool left = x0 < DVFE_PADX;                         // pixels x0+1 .. x0+8 -> x' = -x0-8 .. -x0-1
    const int q8 = D.w - 8 - x0;                              // right: pixels x0-1 .. x0+6 -> x' = w+q8 .. w+q8+7
    const bool right = q8 < padR;
    // border word at x' in [-4j-4, -4j-1] = bytes (W[j+1].b0, W[j].b3, W[j].b2, W[j].b1); at [w+4m, w+4m+3] = (W'[m].b2, b1, b0, W'[m+1].b3)
    const uint2 lb = make_uint2(__byte_perm(v.y, nxt, 0x1234), __byte_perm(v.x, v.y, 0x1234));
    const uint2 rb = make_uint2(__byte_perm(v.y, v.x, 0x7012), __byte_perm(v.x, prv, 0x7012));
    int ys[3], ny = 1;
    ys[0] = y;
    if (y >= 1 && y <= DVFE_PADY) ys[ny++] = -y;
    if (y <= D.h - 2 && y >= D.h - 1 - DVFE_PADY) ys[ny++] = 2 * (D.h - 1) - y;
    for (int j = 0; j < ny; j++) {
        uint8_t* __restrict__ row = dst + (ptrdiff_t)ys[j] * D.pitch;
        *reinterpret_cast<uint2*>(row + x0) = v;
        if (left) *reinterpret_cast<uint2*>(row - x0 - 8) = lb;
        if (right) *reinterpret_cast<uint2*>(row + D.w + q8) = rb;
    }
}

// one thread = 8 consecutive outputs of two consecutive rows.  It reads 7 source rows (one 16-byte and two
// 4-byte aligned loads each) and evaluates the separable 5x5 kernel with dp4a: the horizontal taps (1 4 6 4)
// times the vertical weight fit int8, the fifth tap is a second dp4a.  fuse_border: also store the level's border (above).
__device__ __forceinline__ void pyr_down_body(uint8_t* base, const PyrLevel& S, const PyrLevel& D, int x0, int y0, bool fuse_border) {
    const uint8_t* __restrict__ src = base + S.offset + (size_t)DVFE_PADY * S.pitch + DVFE_PADX;   // pixel (0,0)
    uint8_t* __restrict__ dst = base + D.offset + (size_t)DVFE_PADY * D.pitch + DVFE_PADX;
    if (x0 >= D.w || y0 >= D.h) return;
    if (x0 + 7 < D.w && y0 + 1 < D.h) {
        unsigned acc0[8], acc1[8];
#pragma unroll
        for (int j = 0; j < 8; j++) { acc0[j] = 128u; acc1[j] = 128u; }
        // source rows 2*y0-2 .. 2*y0+4 ; output row 0 uses rows 0..4, output row 1 uses rows 2..6
#pragma unroll
        for (int r = 0; r < 7; r++) {
            const uint8_t* rp = src + (size_t)(2 * y0 - 2 + r) * S.pitch + 2 * x0;
            unsigned W[6];
            W[0] = __ldg(reinterpret_cast<const unsigned*>(rp - 4));
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(rp));
            W[1] = q.x; W[2] = q.y; W[3] = q.z; W[4] = q.w;
            W[5] = __ldg(reinterpret_cast<const unsigned*>(rp + 16));
            // vertical weight of this source row for each output row (0 = unused)
            const int k0 = (r == 0 || r == 4) ? 1 : (r == 1 || r == 3) ? 4 : (r == 2) ? 6 : 0;
            const int k1 = (r == 2 || r == 6) ? 1 : (r == 3 || r == 5) ? 4 : (r == 4) ? 6 : 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int m = j >> 1;
                unsigned A, E;     // A: bytes [2j-2, 2j+2) ; E: word holding byte 2j+2
                unsigned esel;     // weight position of byte 2j+2 inside E
                if ((j & 1) == 0) { A = __funnelshift_r(W[m], W[m + 1], 16); E = W[m + 1]; esel = 16; }
                else { A = W[m + 1]; E = W[m + 2]; esel = 0; }
                if (k0) {
                    acc0[j] = __dp4a(A, (unsigned)(k0 * 0x04060401), acc0[j]);
                    acc0[j] = __dp4a(E, (unsigned)k0 << esel, acc0[j]);
                }
                if (k1) {
                    acc1[j] = __dp4a(A, (unsigned)(k1 * 0x04060401), acc1[j]);
                    acc1[j] = __dp4a(E, (unsigned)k1 << esel, acc1[j]);
                }
            }
        }
        uint2 o0, o1;
        o0.x = (acc0[0] >> 8) | ((acc0[1] >> 8) << 8) | ((acc0[2] >> 8) << 16) | ((acc0[3] >> 8) << 24);
        o0.y = (acc0[4] >> 8) | ((acc0[5] >> 8) << 8) | ((acc0[6] >> 8) << 16) | ((acc0[7] >> 8) << 24);
        o1.x = (acc1[0] >> 8) | ((acc1[1] >> 8) << 8) | ((acc1[2] >> 8) << 16) | ((acc1[3] >> 8) << 24);
        o1.y = (acc1[4] >> 8) | ((acc1[5] >> 8) << 8) | ((acc1[6] >> 8) << 16) | ((acc1[7] >> 8) << 24);
        if (!fuse_border) {
            *reinterpret_cast<uint2*>(dst + (size_t)y0 * D.pitch + x0) = o0;
            *reinterpret_cast<uint2*>(dst + (size_t)(y0 + 1) * D.pitch + x0) = o1;
            return;
        }
        // the neighbours' adjacent words (the lanes of a warp are consecutive x0 of one row pair; w % 8 == 0, so every lane that
        // has pixels is here)
        const unsigned am = __activemask();
        const unsigned n0 = __shfl_down_sync(am, o0.x, 1), n1 = __shfl_down_sync(am, o1.x, 1);
        const unsigned p0 = __shfl_up_sync(am, o0.y, 1), p1 = __shfl_up_sync(am, o1.y, 1);
        const bool edge = x0 < DVFE_PADX || D.w - 8 - x0 < D.pitch - DVFE_PADX - D.w || y0 <= DVFE_PADY || y0 + 1 >= D.h - 1 - DVFE_PADY;
        if (!edge) {
            *reinterpret_cast<uint2*>(dst + (size_t)y0 * D.pitch + x0) = o0;
            *reinterpret_cast<uint2*>(dst + (size_t)(y0 + 1) * D.pitch + x0) = o1;
            return;
        }
        pyr_store8_fused(dst, D, x0, y0, o0, n0, p0);
        pyr_store8_fused(dst, D, x0, y0 + 1, o1, n1, p1);
        return;
    }
    // the ragged right / bottom edge of the interior (w % 8, odd h)
    for (int rr = 0; rr < 2 && y0 + rr < D.h; rr++)
        for (int i = 0; i < 8 && x0 + i < D.w; i++) {
            const uint8_t* c = src + (size_t)(2 * (y0 + rr)) * S.pitch + 2 * (x0 + i);
            const int s = pyr_tap5(c - 2 * S.pitch) + 4 * pyr_tap5(c - S.pitch) + 6 * pyr_tap5(c) +
                          4 * pyr_tap5(c + S.pitch) + pyr_tap5(c + 2 * S.pitch);
            const uint8_t v = (uint8_t)((s + 128) >> 8);
            if (fuse_border) pyr_store_px_mirrored(dst, D, x0 + i, y0 + rr, v);
            else dst[(size_t)(y0 + rr) * D.pitch + x0 + i] = v;
        }
}

// fuse_border != 0: the level's REFLECT_101 border is stored here too (no k_pyr_border launch for it)
__global__ void __launch_bounds__(256, 5) k_pyr_down(PyrImgSet set, PyrLevel S, PyrLevel D, int fuse_border) {
    const uint8_t* unused; uint8_t* base;
    pyr_select(set, blockIdx.z, unused, base);
    pyr_down_body(base, S, D, (blockIdx.x * blockDim.x + threadIdx.x) * 8, (blockIdx.y * blockDim.y + threadIdx.y) * 2, fuse_border != 0);
}

__global__ void __launch_bounds__(256) k_pyr_down_jobs(const PyrJob* __restrict__ jobs, int level) {
    const PyrJob& J = jobs[blockIdx.z];
    if (level >= J.desc.n_levels) return;
    pyr_down_body(J.dst, J.desc.lv[level - 1], J.desc.lv[level], (blockIdx.x * blockDim.x + threadIdx.x) * 8,
                  (blockIdx.y * blockDim.y + threadIdx.y) * 2, false);
}

// level 0 of a job: the source image (sw x sh) zero-extended at the bottom/right to the level size
// (InstanceImagePadding: cv::copyMakeBorder(..., BORDER_CONSTANT, 0), front_end/feature_utils.cpp:406-413)
__global__ void __launch_bounds__(256) k_pyr_level0_jobs(const PyrJob* __restrict__ jobs) {
    const PyrJob& J = jobs[blockIdx.z];
    const PyrLevel L = J.desc.lv[0];
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= L.w || y >= L.h) return;
    uint8_t v = 0;
    if (x < J.sw && y < J.sh) v = J.src[(size_t)y * J.spitch + x];
    J.dst[L.offset + (size_t)(y + DVFE_PADY) * L.pitch + DVFE_PADX + x] = v;
}

int launch_build_pyramids_jobs(const PyrJob* d_jobs, int n_jobs, int max_w, int max_h, int max_levels, cudaStream_t st) {
    if (n_jobs <= 0) return DVFE_OK;
    const dim3 blk(32, 8);
    {
        dim3 grid((max_w + 31) / 32, (max_h + 7) / 8, n_jobs);
        DVFE_LAUNCH(k_pyr_level0_jobs, grid, blk, 0, st, d_jobs);
    }
    int w = max_w, h = max_h;
    for (int l = 0; l < max_levels; l++) {
        if (l > 0) {
            w = (w + 1) / 2; h = (h + 1) / 2;
            dim3 grid(((w + 7) / 8 + 31) / 32, ((h + 1) / 2 + 7) / 8, n_jobs);
            DVFE_LAUNCH(k_pyr_down_jobs, grid, blk, 0, st, d_jobs, l);
        }
        dim3 bgrid((h + 2 * DVFE_PADY + 7) / 8, 1, n_jobs);
        DVFE_LAUNCH(k_pyr_border_jobs, bgrid, blk, 0, st, d_jobs, l);
    }
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

// crop of a rectangle out of a pitched image into a dense buffer (SemanticImage::SetMaskAndRoi: gray0(rect))
__global__ void __launch_bounds__(256) k_crop_jobs(const CropJob* __restrict__ jobs) {
    const CropJob& J = jobs[blockIdx.z];
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= J.w || y >= J.h) return;
    J.dst[(size_t)y * J.w + x] = J.src[(size_t)(J.y + y) * J.spitch + J.x + x];
}

int launch_crop_jobs(const CropJob* d_jobs, int n_jobs, int max_w, int max_h, cudaStream_t st) {
    if (n_jobs <= 0) return DVFE_OK;
    dim3 blk(32, 8), grid((max_w + 31) / 32, (max_h + 7) / 8, n_jobs);
    DVFE_LAUNCH(k_crop_jobs, grid, blk, 0, st, d_jobs);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

// the caller's dense images -> level 0 of the padded pyramids; *border_done (nullable) = the border was written too
static bool pyr_fuse_enabled() {
    static const bool on = []() { const char* e = getenv("DVFE_PYR_FUSE"); return e == nullptr || atoi(e) != 0; }();
    return on;
}
bool pyr_level0_writes_border(const PyrDesc& desc) { return pyr_fuse_enabled() && pyr_level0_fusable(desc.lv[0]); }

int launch_pyr_level0(const PyrImgSet& set, int n_img, const PyrDesc& desc, int spitch, cudaStream_t st) {
    const dim3 blk(32, 8);
    const PyrLevel& L = desc.lv[0];
    dim3 grid(((L.w + 15) / 16 + 31) / 32, (L.h + 7) / 8, n_img);
    DVFE_LAUNCH(k_pyr_level0, grid, blk, 0, st, set, L, spitch, pyr_level0_writes_border(desc) ? 1 : 0);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

int launch_pyr_level0_table(const ImgSrc* d_src, uint8_t* dst, size_t dst_stride, int n_img, const PyrDesc& desc, cudaStream_t st) {
    const PyrLevel& L = desc.lv[0];
    dim3 grid(((L.w + 15) / 16 + 31) / 32, (L.h + 7) / 8, n_img);
    DVFE_LAUNCH(k_pyr_level0_table, grid, dim3(32, 8), 0, st, d_src, dst, dst_stride, L, pyr_level0_writes_border(desc) ? 1 : 0);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

// level0_mode: DVFE_L0_BUILD = copy level 0 from set.src; DVFE_L0_INTERIOR = its interior is in place (H2D straight into the padded
// layout, or an ingest kernel), the border is not; DVFE_L0_COMPLETE = interior and border are in place
int launch_build_pyramids(const PyrImgSet& set, int n_img, const PyrDesc& desc, int spitch, cudaStream_t st, int level0_mode) {
    const dim3 blk(32, 8);
    bool l0_border_done = level0_mode == DVFE_L0_COMPLETE;
    if (level0_mode == DVFE_L0_BUILD) {
        const int rc = launch_pyr_level0(set, n_img, desc, spitch, st);
        if (rc != DVFE_OK) return rc;
        l0_border_done = pyr_level0_writes_border(desc);
    }
    for (int l = 0; l < desc.n_levels; l++) {
        const PyrLevel& D = desc.lv[l];
        // levels >= 1 store their own border from the down-sampling kernel; levels too small or too ragged for single word
        // reflections keep a border launch
        const bool fuse = l > 0 && pyr_fuse_enabled() && pyr_border_fusable(D);
        if (l > 0) {
            dim3 grid(((D.w + 7) / 8 + 31) / 32, ((D.h + 1) / 2 + 7) / 8, n_img);
            DVFE_LAUNCH(k_pyr_down, grid, blk, 0, st, set, desc.lv[l - 1], D, fuse ? 1 : 0);
        }
        if (!fuse && !(l == 0 && l0_border_done)) launch_pyr_border(set, n_img, D, st);
    }
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

// unpadded copy of one level back out (seam op dvfe_op_build_pyramid)
__global__ void k_pyr_extract(const uint8_t* base, PyrLevel L, uint8_t* out) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= L.w || y >= L.h) return;
    out[(size_t)y * L.w + x] = base[L.offset + (size_t)(y + DVFE_PADY) * L.pitch + DVFE_PADX + x];
}

// one level with `border` pixels of its REFLECT_101 border on every side, dense (w + 2 border) x (h + 2 border)
__global__ void k_pyr_extract_bordered(const uint8_t* base, PyrLevel L, int border, uint8_t* out) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int ow = L.w + 2 * border, oh = L.h + 2 * border;
    if (x >= ow || y >= oh) return;
    out[(size_t)y * ow + x] = base[L.offset + (size_t)(y - border + DVFE_PADY) * L.pitch + DVFE_PADX + x - border];
}

int launch_pyr_extract_bordered(const uint8_t* pyr, const PyrLevel& L, int border, uint8_t* out, cudaStream_t st) {
    dim3 blk(32, 8), grid((L.w + 2 * border + 31) / 32, (L.h + 2 * border + 7) / 8);
    DVFE_LAUNCH(k_pyr_extract_bordered, grid, blk, 0, st, pyr, L, border, out);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}

int launch_pyr_extract(const uint8_t* pyr, const PyrLevel& L, uint8_t* out, cudaStream_t st) {
    dim3 blk(32, 8), grid((L.w + 31) / 32, (L.h + 7) / 8);
    DVFE_LAUNCH(k_pyr_extract, grid, blk, 0, st, pyr, L, out);
    DVFE_CUDA(cudaGetLastError());
    return DVFE_OK;
}
