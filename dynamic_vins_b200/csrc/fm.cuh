// Device helpers of cv::findFundamentalMat(FM_RANSAC) shared by the seam op (geometry.cu, k_reject_with_f) and the in-step
// rejection (reject.cu, k_reject_with_f_step): the cv::RNG stream, the 7-point solver, the collinearity test of a sample, the
// per-correspondence error and RANSACUpdateNumIters, all fp64 in the operation order of the OpenCV source (the library is built
// -fmad=false, so both kernels compute the same bits).
#pragma once
#include "kernels.cuh"

#define FM_MODEL_POINTS 7
#define FM_MAX_ITERS 1000       // cv::findFundamentalMat's maxIters

namespace {

struct FmRng {                  // cv::RNG: multiply-with-carry
    unsigned long long state;
    __device__ unsigned next() {
        state = (unsigned long long)(unsigned)state * 4164903690ull + (unsigned)(state >> 32);
        return (unsigned)state;
    }
    __device__ int uniform(int a, int b) { return a == b ? a : (int)(next() % (unsigned)(b - a) + a); }
};

__device__ int fm_solve_cubic(const double* c, double* x) {          // cv::solveCubic
    double a0 = c[0], a1 = c[1], a2 = c[2], a3 = c[3];
    if (a0 == 0) {
        if (a1 == 0) {
            if (a2 == 0) return a3 == 0 ? -1 : 0;
            x[0] = -a3 / a2;
            return 1;
        }
        double d = a2 * a2 - 4 * a1 * a3;
        if (d >= 0) {
            d = sqrt(d);
            const double q1 = (-a2 + d) * 0.5, q2 = (a2 + d) * -0.5;
            if (fabs(q1) > fabs(q2)) { x[0] = q1 / a1; x[1] = a3 / q1; }
            else { x[0] = q2 / a1; x[1] = a3 / q2; }
            return d > 0 ? 2 : 1;
        }
        return 0;
    }
    a0 = 1. / a0; a1 *= a0; a2 *= a0; a3 *= a0;
    const double Q = (a1 * a1 - 3 * a2) * (1. / 9);
    const double R = (2 * a1 * a1 * a1 - 9 * a1 * a2 + 27 * a3) * (1. / 54);
    const double Qcubed = Q * Q * Q;
    double d = Qcubed - R * R;
    if (d > 0) {
        const double theta = acos(R / sqrt(Qcubed));
        const double sqrtQ = sqrt(Q);
        const double t0 = -2 * sqrtQ, t1 = theta * (1. / 3), t2 = a1 * (1. / 3);
        x[0] = t0 * cos(t1) - t2;
        x[1] = t0 * cos(t1 + (2. * 3.1415926535897932384626433832795 / 3)) - t2;
        x[2] = t0 * cos(t1 + (4. * 3.1415926535897932384626433832795 / 3)) - t2;
        return 3;
    }
    if (d == 0) {
        if (R >= 0) { x[0] = -2 * pow(R, 1. / 3) - a1 / 3; x[1] = pow(R, 1. / 3) - a1 / 3; }
        else { x[0] = 2 * pow(-R, 1. / 3) - a1 / 3; x[1] = -pow(-R, 1. / 3) - a1 / 3; }
        return x[0] == x[1] ? 1 : 2;
    }
    d = sqrt(-d);
    double e = pow(d + fabs(R), 1. / 3);
    if (R > 0) e = -e;
    x[0] = (e + Q / e) - a1 * (1. / 3);
    return 1;
}

// Null space of the 7 x 9 epipolar system by Gauss-Jordan elimination with complete pivoting; f1 / f2 = the solutions with the
// two free unknowns set to (1, 0) / (0, 1).  (OpenCV takes an orthonormal basis from its SVD; the set of F's is the same.)
__device__ bool fm_null_space(double (*A)[9], double* f1, double* f2) {
    int perm[9];
    for (int j = 0; j < 9; j++) perm[j] = j;
    for (int k = 0; k < 7; k++) {
        int pr = k, pc = k;
        double best = -1.0;
        for (int i = k; i < 7; i++)
            for (int j = k; j < 9; j++)
                if (fabs(A[i][j]) > best) { best = fabs(A[i][j]); pr = i; pc = j; }
        if (!(best > 0.0)) return false;
        if (pr != k) for (int j = 0; j < 9; j++) { const double t = A[k][j]; A[k][j] = A[pr][j]; A[pr][j] = t; }
        if (pc != k) {
            for (int i = 0; i < 7; i++) { const double t = A[i][k]; A[i][k] = A[i][pc]; A[i][pc] = t; }
            const int t = perm[k]; perm[k] = perm[pc]; perm[pc] = t;
        }
        const double inv = 1.0 / A[k][k];
        for (int j = k; j < 9; j++) A[k][j] *= inv;
        for (int i = 0; i < 7; i++) {
            if (i == k) continue;
            const double m = A[i][k];
            if (m == 0.0) continue;
            for (int j = k; j < 9; j++) A[i][j] -= m * A[k][j];
        }
    }
    for (int i = 0; i < 7; i++) { f1[perm[i]] = -A[i][7]; f2[perm[i]] = -A[i][8]; }
    f1[perm[7]] = 1.0; f1[perm[8]] = 0.0;
    f2[perm[7]] = 0.0; f2[perm[8]] = 1.0;
    return true;
}

// run7Point on the sample (m1[idx], m2[idx]): up to 3 fundamental matrices, each scaled to F[8] = 1
__device__ int fm_run7(const float2* __restrict__ m1, const float2* __restrict__ m2, const int* idx, double* F) {
    double A[7][9], f1[9], f2[9], c[4], r[3] = {0, 0, 0};
    for (int i = 0; i < 7; i++) {
        const float2 a = m1[idx[i]], b = m2[idx[i]];
        const double x0 = a.x, y0 = a.y, x1 = b.x, y1 = b.y;
        A[i][0] = x1 * x0; A[i][1] = x1 * y0; A[i][2] = x1;
        A[i][3] = y1 * x0; A[i][4] = y1 * y0; A[i][5] = y1;
        A[i][6] = x0; A[i][7] = y0; A[i][8] = 1;
    }
    if (!fm_null_space(A, f1, f2)) return 0;
    for (int i = 0; i < 9; i++) f1[i] -= f2[i];
    double t0 = f2[4] * f2[8] - f2[5] * f2[7], t1 = f2[3] * f2[8] - f2[5] * f2[6], t2 = f2[3] * f2[7] - f2[4] * f2[6];
    c[3] = f2[0] * t0 - f2[1] * t1 + f2[2] * t2;
    c[2] = f1[0] * t0 - f1[1] * t1 + f1[2] * t2 - f1[3] * (f2[1] * f2[8] - f2[2] * f2[7]) + f1[4] * (f2[0] * f2[8] - f2[2] * f2[6]) -
           f1[5] * (f2[0] * f2[7] - f2[1] * f2[6]) + f1[6] * (f2[1] * f2[5] - f2[2] * f2[4]) - f1[7] * (f2[0] * f2[5] - f2[2] * f2[3]) +
           f1[8] * (f2[0] * f2[4] - f2[1] * f2[3]);
    t0 = f1[4] * f1[8] - f1[5] * f1[7]; t1 = f1[3] * f1[8] - f1[5] * f1[6]; t2 = f1[3] * f1[7] - f1[4] * f1[6];
    c[0] = f1[0] * t0 - f1[1] * t1 + f1[2] * t2;
    c[1] = f2[0] * t0 - f2[1] * t1 + f2[2] * t2 - f2[3] * (f1[1] * f1[8] - f1[2] * f1[7]) + f2[4] * (f1[0] * f1[8] - f1[2] * f1[6]) -
           f2[5] * (f1[0] * f1[7] - f1[1] * f1[6]) + f2[6] * (f1[1] * f1[5] - f1[2] * f1[4]) - f2[7] * (f1[0] * f1[5] - f1[2] * f1[3]) +
           f2[8] * (f1[0] * f1[4] - f1[1] * f1[3]);
    const int n = fm_solve_cubic(c, r);
    if (n < 1 || n > 3) return 0;
    for (int k = 0; k < n; k++, F += 9) {
        double lambda = r[k], mu = 1.;
        const double s = f1[8] * r[k] + f2[8];
        if (fabs(s) > 2.220446049250313e-16) { mu = 1. / s; lambda *= mu; F[8] = 1.; }
        else F[8] = 0.;
        for (int i = 0; i < 8; i++) F[i] = f1[i] * lambda + f2[i] * mu;
    }
    return n;
}

// haveCollinearPoints on the sample: only its last point is tested against the pairs before it
__device__ bool fm_collinear(const float2* __restrict__ m, const int* idx) {
    const float2 pi = m[idx[6]];
    for (int j = 0; j < 6; j++) {
        const float2 pj = m[idx[j]];
        const double dx1 = pj.x - pi.x, dy1 = pj.y - pi.y;      // float subtraction widened, as `double dx1 = ptr[j].x - ptr[i].x`
        for (int k = 0; k < j; k++) {
            const float2 pk = m[idx[k]];
            const double dx2 = pk.x - pi.x, dy2 = pk.y - pi.y;
            if (fabs(dx2 * dy1 - dy2 * dx1) <= 1.1920928955078125e-07 * (fabs(dx1) + fabs(dy1) + fabs(dx2) + fabs(dy2))) return true;
        }
    }
    return false;
}

// FMEstimatorCallback::computeError of one correspondence (symmetric squared epipolar distance, narrowed to float)
__device__ __forceinline__ float fm_error(const double* F, float2 p1, float2 p2) {
    const double x1 = p1.x, y1 = p1.y, x2 = p2.x, y2 = p2.y;
    double a = F[0] * x1 + F[1] * y1 + F[2], b = F[3] * x1 + F[4] * y1 + F[5], c = F[6] * x1 + F[7] * y1 + F[8];
    const double s2 = 1. / (a * a + b * b), d2 = x2 * a + y2 * b + c;
    a = F[0] * x2 + F[3] * y2 + F[6]; b = F[1] * x2 + F[4] * y2 + F[7]; c = F[2] * x2 + F[5] * y2 + F[8];
    const double s1 = 1. / (a * a + b * b), d1 = x1 * a + y1 * b + c;
    const double e1 = d1 * d1 * s1, e2 = d2 * d2 * s2;
    return (float)(e1 > e2 ? e1 : e2);
}

__device__ int fm_update_iters(double p, double ep, int model_points, int max_iters) {      // RANSACUpdateNumIters
    p = p > 0. ? p : 0.; p = p < 1. ? p : 1.;
    ep = ep > 0. ? ep : 0.; ep = ep < 1. ? ep : 1.;
    double num = 1. - p > 2.2250738585072014e-308 ? 1. - p : 2.2250738585072014e-308;
    double denom = 1. - pow(1. - ep, (double)model_points);
    if (denom < 2.2250738585072014e-308) return 0;
    num = log(num); denom = log(denom);
    return denom >= 0 || -num >= max_iters * (-denom) ? max_iters : (int)llrint(num / denom);
}

// RejectWithF's lifting of one distorted pixel (PinholeCamera::liftProjective, fp64) and re-projection with the virtual focal
// length 460 about the image centre, narrowed to float as cv::Point2f((float)x, (float)y)
__device__ __forceinline__ float2 fm_reproject(const CamParams& cam, float2 p, double half_col, double half_row) {
    const double u = (double)p.x, v = (double)p.y;
    const double mx_d = cam.inv_K11 * u + cam.inv_K13, my_d = cam.inv_K22 * v + cam.inv_K23;
    double mx_u = mx_d, my_u = my_d;
    if (!cam.no_distortion) {
#pragma unroll 1
        for (int it = 0; it < 8; it++) {
            const double x = mx_u, y = my_u;
            const double mx2 = x * x, my2 = y * y, mxy = x * y, rho2 = mx2 + my2;
            const double rad = cam.k1 * rho2 + cam.k2 * rho2 * rho2;
            const double dux = x * rad + 2.0 * cam.p1 * mxy + cam.p2 * (rho2 + 2.0 * mx2);
            const double duy = y * rad + 2.0 * cam.p2 * mxy + cam.p1 * (rho2 + 2.0 * my2);
            mx_u = mx_d - dux; my_u = my_d - duy;
        }
    }
    return make_float2((float)(460.0 * mx_u / 1.0 + half_col), (float)(460.0 * my_u / 1.0 + half_row));
}

}  // namespace
