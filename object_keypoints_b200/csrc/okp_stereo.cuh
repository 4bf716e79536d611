// okp_stereo.cuh -- two-view stereo helpers, one thread per point pair, float64 in registers.
//
//   okp_correct_matches_kernel   cv2.correctMatches as StereoCamera.triangulate calls it
//                                (perception/utils/camera_utils.py:100-101): the Hartley-Sturm
//                                optimal correction (Hartley & Zisserman, Alg. 12.1). Moves a
//                                pair (x, x') by the smallest total squared distance onto a pair
//                                that satisfies x'^T F x = 0 exactly.
//   okp_associate_kernel         stereo association by epipolar distance, one-to-one, -1 for
//                                unmatched; the implementation is gone from the reference, its
//                                expectations survive in test/test_pipeline.py:208-261.
//
// The correction is geometric (a unique global minimum of a rational cost over one real
// parameter t), so any exact minimiser reproduces OpenCV's output. OpenCV finds the stationary
// points as the six roots of a degree-6 polynomial g(t) with a Durand-Kerner iteration; here the
// roots come from an Aberth-Ehrlich iteration started on the Newton polygon of the coefficients
// (so that roots of very different magnitude -- the epipole of a sideways stereo rig is ~1e6 px
// away -- all start at the right scale), the cost is evaluated at the real part of every root and
// at t = infinity like OpenCV does, and the winner is polished by Newton steps on g.
#pragma once
#include "okp_common.cuh"

struct OkpMat3 { double m[9]; };

// Unit right singular vector of the smallest singular value of the 3x3 matrix A (destroyed):
// one-sided (Hestenes) Jacobi, the same scheme as the 4x4 solve of okp_dlt.cuh.
__host__ __device__ __forceinline__ void okp_null_vector3(double (&A)[3][3], double (&h)[3]) {
    double Vm[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    for (int sweep = 0; sweep < 60; ++sweep) {
        bool rotated = false;
#pragma unroll
        for (int p = 0; p < 2; ++p) {
#pragma unroll
            for (int q = p + 1; q < 3; ++q) {
                double alpha = 0, beta = 0, gamma = 0;
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    alpha += A[r][p] * A[r][p];
                    beta += A[r][q] * A[r][q];
                    gamma += A[r][p] * A[r][q];
                }
                if (fabs(gamma) <= 1e-300 || fabs(gamma) <= 2.3e-16 * sqrt(alpha * beta)) continue;
                rotated = true;
                const double zeta = (beta - alpha) / (2.0 * gamma);
                const double tt = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                const double cs = 1.0 / sqrt(1.0 + tt * tt), sn = cs * tt;
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const double ap = A[r][p], aq = A[r][q];
                    A[r][p] = cs * ap - sn * aq;
                    A[r][q] = sn * ap + cs * aq;
                    const double vp = Vm[r][p], vq = Vm[r][q];
                    Vm[r][p] = cs * vp - sn * vq;
                    Vm[r][q] = sn * vp + cs * vq;
                }
            }
        }
        if (!rotated) break;
    }
    int arg = 0;
    double smallest = 0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        double nrm = 0;
#pragma unroll
        for (int r = 0; r < 3; ++r) nrm += A[r][c] * A[r][c];
        if (c == 0 || nrm < smallest) { smallest = nrm; arg = c; }
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) h[r] = arg == 0 ? Vm[r][0] : (arg == 1 ? Vm[r][1] : Vm[r][2]);
}

struct OkpComplex { double re, im; };
__host__ __device__ __forceinline__ OkpComplex okp_cmul(OkpComplex a, OkpComplex b) {
    return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re};
}
__host__ __device__ __forceinline__ OkpComplex okp_cdiv(OkpComplex a, OkpComplex b) {      // Smith's algorithm
    // branch-free (selects): the two cases of the textbook form differ by which component of b is the pivot; with
    // p = pivot, q = the other one, x / y = the matching components of a, both cases are ((x + y r) / den, +-(y - x r) / den)
    // -- the same operations on the same operands as the two-branch form, so the quotient is bit-identical, and the lanes
    // of a warp no longer split on |b.re| >= |b.im|
    const bool big = fabs(b.re) >= fabs(b.im);
    const double p = big ? b.re : b.im, q = big ? b.im : b.re;
    const double x = big ? a.re : a.im, y = big ? a.im : a.re;
    const double r = q / p, den = p + q * r;
    const double im = (y - x * r) / den;
    return {(x + y * r) / den, big ? im : -im};
}

// All complex roots of k[0] + k[1] t + ... + k[6] t^6 (degree n <= 6 after leading zeros are
// dropped). Returns n. Aberth-Ehrlich, Gauss-Seidel order, start values on the Newton polygon
// (Bini 1996): for every edge (i, j) of the upper convex hull of (i, log|k_i|), j - i roots on a
// circle of radius |k_i / k_j|^(1 / (j - i)).
__host__ __device__ __noinline__ int okp_poly6_roots(const double* k, OkpComplex* z) {
    int n = 6;
    while (n > 0 && k[n] == 0.0) --n;
    if (n == 0) return 0;
    double lg[7];
    for (int i = 0; i <= n; ++i) lg[i] = k[i] != 0.0 ? log(fabs(k[i])) : -1e300;
    int placed = 0, i = 0;
    while (i < n) {
        int best = i + 1;
        double slope = (lg[i + 1] - lg[i]);
        for (int j = i + 2; j <= n; ++j) {
            const double s = (lg[j] - lg[i]) / (double)(j - i);
            if (s >= slope) { slope = s; best = j; }
        }
        const int m = best - i;
        double radius = lg[i] <= -1e299 ? 0.0 : exp(-slope);
        if (!(radius < 1e150)) radius = 1e150;
        for (int r = 0; r < m; ++r) {
            const double ang = 6.283185307179586 * ((double)r / m + (double)placed / n) + 0.7;
            double sn, cs;
            sincos(ang, &sn, &cs);
            z[placed++] = {radius * cs, radius * sn};
        }
        i = best;
    }
    // Convergence: the largest relative correction of a sweep below 1e-14 -- or no longer contracting once it is small.
    // Aberth-Ehrlich converges cubically, so a sweep that is within 1e-9 of the roots and does not shrink the correction
    // fourfold has reached the rounding floor of an ill-conditioned root (the far roots of a sideways rig sit at |t| ~ 1e6
    // and stall at ~1e-15 .. 1e-13). Round 1 asked every root for 4e-16: one pair in five never got there and ran to the
    // cap of 200 sweeps, and with it the other 31 pairs of its warp (ncu r02m: 4 of 32 lanes active, 19.9 ms per 2^20
    // pairs). The winner is polished by Newton steps on g below, so the result does not move (<= 1e-12 px).
    double previous = 1e300;
    for (int it = 0; it < 200; ++it) {
        double worst = 0.0;
        for (int r = 0; r < n; ++r) {
            const OkpComplex x = z[r];
            OkpComplex p = {k[n], 0.0}, dp = {0.0, 0.0};
            for (int c = n - 1; c >= 0; --c) {
                dp = okp_cmul(dp, x);
                dp.re += p.re; dp.im += p.im;
                p = okp_cmul(p, x);
                p.re += k[c];
            }
            if (p.re == 0.0 && p.im == 0.0) continue;
            OkpComplex w;
            if (dp.re == 0.0 && dp.im == 0.0) {
                w = {1e-3 * (fabs(x.re) + 1e-3), 1e-3 * (fabs(x.im) + 1e-3)};     // stationary point: nudge off it
            } else {
                w = okp_cdiv(p, dp);
                OkpComplex s = {0.0, 0.0};
                for (int j = 0; j < n; ++j) {
                    if (j == r) continue;
                    const OkpComplex d = {x.re - z[j].re, x.im - z[j].im};
                    if (d.re == 0.0 && d.im == 0.0) continue;
                    const OkpComplex inv = okp_cdiv({1.0, 0.0}, d);
                    s.re += inv.re; s.im += inv.im;
                }
                const OkpComplex ws = okp_cmul(w, s);
                const OkpComplex den = {1.0 - ws.re, -ws.im};
                if (den.re != 0.0 || den.im != 0.0) w = okp_cdiv(w, den);
            }
            z[r] = {x.re - w.re, x.im - w.im};
            const double rel = (fabs(w.re) + fabs(w.im)) / (fabs(x.re) + fabs(x.im) + 1e-300);
            if (rel > worst) worst = rel;
        }
        if (worst < 1e-14 || (worst < 1e-9 && worst > 0.25 * previous)) break;
        previous = worst;
    }
    return n;
}

// The epipoles of F itself, once per call (host): right null vector (F e = 0) and left null vector (e^T F = 0).
struct OkpEpipoles { double right[3], left[3]; };
__host__ __device__ __forceinline__ OkpEpipoles okp_epipoles(const OkpMat3& Fm) {
    double B[3][3], Bt[3][3];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) { B[r][c] = Fm.m[3 * r + c]; Bt[r][c] = Fm.m[3 * c + r]; }
    OkpEpipoles e;
    okp_null_vector3(B, e.right);
    okp_null_vector3(Bt, e.left);
    return e;
}

// One pair: Hartley-Sturm correction (__host__ too: tools/host_check_stereo.cu runs it on the CPU
// of the build container, which has no GPU). F row-major with x2^T F x1 = 0.
__host__ __device__ __forceinline__ void okp_correct_pair(const OkpMat3& Fm, const OkpEpipoles& ep, double x1, double y1,
                                                          double x2, double y2, double* o1, double* o2) {
    const double* F = Fm.m;
    // F~ = T2^T F T1 with T = [[1,0,x],[0,1,y],[0,0,1]]: both points move to the origin
    double A[3][3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        A[0][c] = F[c];
        A[1][c] = F[3 + c];
        A[2][c] = x2 * F[c] + y2 * F[3 + c] + F[6 + c];
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) A[r][2] = A[r][0] * x1 + A[r][1] * y1 + A[r][2];
    // epipoles: F~ e1 = 0, e2^T F~ = 0, scaled so that e_x^2 + e_y^2 = 1. F~ = T2^T F T1, so F (T1 e1) = 0 and
    // (T2 e2)^T F = 0: e = T^-1 (epipole of F) -- a translation of F's own epipoles (round 1 ran two 3x3 Jacobi SVDs of F~
    // per pair for them)
    const double e1[3] = {ep.right[0] - x1 * ep.right[2], ep.right[1] - y1 * ep.right[2], ep.right[2]};
    const double e2[3] = {ep.left[0] - x2 * ep.left[2], ep.left[1] - y2 * ep.left[2], ep.left[2]};
    const double s1 = sqrt(e1[0] * e1[0] + e1[1] * e1[1]);
    const double s2 = sqrt(e2[0] * e2[0] + e2[1] * e2[1]);
    const double e1x = e1[0] / s1, e1y = e1[1] / s1, e1z = e1[2] / s1;
    const double e2x = e2[0] / s2, e2y = e2[1] / s2, e2z = e2[2] / s2;
    // F' = R2 F~ R1^T with R = [[ex, ey, 0], [-ey, ex, 0], [0, 0, 1]]: epipoles onto the x axes
    double G[3][3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        G[0][c] = e2x * A[0][c] + e2y * A[1][c];
        G[1][c] = -e2y * A[0][c] + e2x * A[1][c];
        G[2][c] = A[2][c];
    }
    double Fp[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        Fp[r][0] = G[r][0] * e1x + G[r][1] * e1y;
        Fp[r][1] = -G[r][0] * e1y + G[r][1] * e1x;
        Fp[r][2] = G[r][2];
    }
    const double f1 = e1z, f2 = e2z, a = Fp[1][1], b = Fp[1][2], c = Fp[2][1], d = Fp[2][2];
    const double f1_2 = f1 * f1, f1_4 = f1_2 * f1_2, f2_2 = f2 * f2, f2_4 = f2_2 * f2_2;
    const double a2 = a * a, b2 = b * b, c2 = c * c, d2 = d * d;
    // g(t) = t ((a t + b)^2 + f2^2 (c t + d)^2)^2 - (a d - b c)(1 + f1^2 t^2)^2 (a t + b)(c t + d), expanded
    double k[7];
    k[6] = b * c2 * f1_4 * a - a2 * d * f1_4 * c;
    k[5] = f2_4 * c2 * c2 + 2 * a2 * f2_2 * c2 - a2 * d2 * f1_4 + b2 * c2 * f1_4 + a2 * a2;
    k[4] = 4 * a2 * a * b + 2 * b * c2 * f1_2 * a + 4 * f2_4 * c2 * c * d + 4 * a * b * f2_2 * c2 +
           4 * a2 * f2_2 * c * d - 2 * a2 * d * f1_2 * c - a * d2 * f1_4 * b + b2 * c * f1_4 * d;
    k[3] = 6 * a2 * b2 + 6 * f2_4 * c2 * d2 + 2 * b2 * f2_2 * c2 + 2 * a2 * f2_2 * d2 - 2 * a2 * d2 * f1_2 +
           2 * b2 * c2 * f1_2 + 8 * a * b * f2_2 * c * d;
    k[2] = 4 * a * b2 * b + 4 * b2 * f2_2 * c * d + 4 * f2_4 * c * d2 * d - a2 * d * c + b * c2 * a +
           4 * a * b * f2_2 * d2 - 2 * a * d2 * f1_2 * b + 2 * b2 * c * f1_2 * d;
    k[1] = f2_4 * d2 * d2 + b2 * b2 + 2 * b2 * f2_2 * d2 - a2 * d2 + b2 * c2;
    k[0] = -a * d2 * b + b2 * c * d;
    double big = 0.0;
#pragma unroll
    for (int i = 0; i < 7; ++i) big = fmax(big, fabs(k[i]));
    if (big > 0.0) {
#pragma unroll
        for (int i = 0; i < 7; ++i) k[i] /= big;
    }
    OkpComplex z[6];
    const int n = okp_poly6_roots(k, z);
    // cost at t = infinity, then at the real part of every root (OpenCV's selection rule)
    double s_best = 1.0 / f1_2 + c2 / (a2 + f2_2 * c2);
    double t_best = 0.0;
    bool at_infinity = true;
    if (!(s_best == s_best)) s_best = INFINITY;
    for (int i = 0; i < n; ++i) {
        const double t = z[i].re;
        const double u = c * t + d, v = a * t + b;
        const double s = (t * t) / (1.0 + f1_2 * t * t) + (u * u) / (v * v + f2_2 * u * u);
        if (s < s_best) { s_best = s; t_best = t; at_infinity = false; }
    }
    double l1[3], l2[3];
    if (!at_infinity) {
        double t = t_best;
        for (int it = 0; it < 4; ++it) {              // polish: Newton on g, kept only while |g| shrinks
            double g = k[6], dg = 0.0;
            for (int i = 5; i >= 0; --i) { dg = dg * t + g; g = g * t + k[i]; }
            if (dg == 0.0 || g == 0.0) break;
            const double tn = t - g / dg;
            double gn = k[6];
            for (int i = 5; i >= 0; --i) gn = gn * tn + k[i];
            if (!(fabs(gn) < fabs(g))) break;
            t = tn;
        }
        const double u = c * t + d, v = a * t + b;
        // closest points to the origin on l1 = (t f1, 1, -t) and l2 = (-f2 u, v, u)
        l1[0] = t * t * f1; l1[1] = t; l1[2] = t * t * f1_2 + 1.0;
        l2[0] = f2 * u * u; l2[1] = -v * u; l2[2] = f2_2 * u * u + v * v;
    } else {                                           // t -> infinity: the limits of the expressions above
        l1[0] = f1; l1[1] = 0.0; l1[2] = f1_2;
        l2[0] = f2 * c2; l2[1] = -a * c; l2[2] = f2_2 * c2 + a2;
    }
    const double p1x = l1[0] / l1[2], p1y = l1[1] / l1[2];
    const double p2x = l2[0] / l2[2], p2y = l2[1] / l2[2];
    // back through R^T and the translations
    o1[0] = e1x * p1x - e1y * p1y + x1;
    o1[1] = e1y * p1x + e1x * p1y + y1;
    o2[0] = e2x * p2x - e2y * p2y + x2;
    o2[1] = e2y * p2x + e2x * p2y + y2;
}

__global__ void __launch_bounds__(64)
okp_correct_matches_kernel(OkpMat3 F, OkpEpipoles ep, const double* __restrict__ left, const double* __restrict__ right, int n,
                           int round_to_f32, double* __restrict__ left_out, double* __restrict__ right_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double o1[2], o2[2];
    okp_correct_pair(F, ep, left[2 * i], left[2 * i + 1], right[2 * i], right[2 * i + 1], o1, o2);
    if (round_to_f32) {                               // OpenCV returns the input dtype (float32 in camera_utils.py:93-101)
        o1[0] = (double)(float)o1[0]; o1[1] = (double)(float)o1[1];
        o2[0] = (double)(float)o2[0]; o2[1] = (double)(float)o2[1];
    }
    left_out[2 * i] = o1[0]; left_out[2 * i + 1] = o1[1];
    right_out[2 * i] = o2[0]; right_out[2 * i + 1] = o2[1];
}

// ---------------------------------------------------------------------------------------------
// Association. One warp per frame pair. cost(i, j) = mean of the two point-to-epipolar-line
// distances (pixels) of UNDISTORTED points, x_R^T F x_L = 0. Greedy one-to-one: repeatedly take
// the globally smallest remaining cost (ties: smallest left index, then smallest right index)
// until it exceeds max_distance. Statement of record: oracle/np_oracle.py::associate.
// okp_associate_kernel and okp_stereo_objects_kernel share the cost and the greedy step below.
// ---------------------------------------------------------------------------------------------
#define OKP_ASSOC_MAX 64

__device__ __forceinline__ double okp_epipolar_cost(const double* F, double x, double y, double xp, double yp) {
    const double l0 = F[0] * x + F[1] * y + F[2], l1 = F[3] * x + F[4] * y + F[5], l2 = F[6] * x + F[7] * y + F[8];
    const double m0 = F[0] * xp + F[3] * yp + F[6], m1 = F[1] * xp + F[4] * yp + F[7];
    const double r = fabs(xp * l0 + yp * l1 + l2);
    return 0.5 * (r / sqrt(l0 * l0 + l1 * l1) + r / sqrt(m0 * m0 + m1 * m1));
}

// The greedy one-to-one step on the costs s_cost[i * stride + j] (i < nl, j < nr <= 64), run by all 32 lanes of a warp.
// The caller clears s_used_left / s_used_right and syncs the warp first. Lane 0 calls on_match(i, j, cost) for every
// match, in the order the matches are taken.
template <typename OnMatch>
__device__ __forceinline__ void okp_greedy_match(const double* s_cost, int stride, int nl, int nr, double max_distance,
                                                 unsigned long long& s_used_left, unsigned long long& s_used_right,
                                                 int lane, OnMatch on_match) {
    const int rounds = nl < nr ? nl : nr;
    for (int round = 0; round < rounds; ++round) {
        const unsigned long long ul = s_used_left, ur = s_used_right;
        double best = INFINITY;
        int arg = 0x7fffffff;
        for (int e = lane; e < nl * nr; e += 32) {
            const int i = e / nr, j = e - i * nr;
            if (((ul >> i) & 1ull) || ((ur >> j) & 1ull)) continue;
            const double c = s_cost[i * stride + j];
            if (c < best || (c == best && e < arg)) { best = c; arg = e; }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, off);
            const int oa = __shfl_xor_sync(0xffffffffu, arg, off);
            if (ob < best || (ob == best && oa < arg)) { best = ob; arg = oa; }
        }
        if (!(best <= max_distance)) break;
        const int i = arg / nr, j = arg - i * nr;
        if (lane == 0) {
            on_match(i, j, best);
            s_used_left = ul | (1ull << i);
            s_used_right = ur | (1ull << j);
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(32)
okp_associate_kernel(OkpMat3 Fm, const double* __restrict__ F_pairs, const double* __restrict__ left,
                     const int32_t* __restrict__ n_left, const double* __restrict__ right,
                     const int32_t* __restrict__ n_right, int ML, int MR, double max_distance,
                     int32_t* __restrict__ match, double* __restrict__ match_cost) {
    extern __shared__ double s_cost[];               // [ML][MR]
    __shared__ unsigned long long s_used_left, s_used_right;
    const int b = blockIdx.x, lane = threadIdx.x;
    const int nl = okp_clamp(n_left[b], 0, ML), nr = okp_clamp(n_right[b], 0, MR);
    // one F for every pair (a stereo rig) or one per pair (two frames of a moving camera: scripts/label.py:285-305)
    const double* F = F_pairs ? F_pairs + 9 * (size_t)b : Fm.m;
    const double* L = left + (size_t)b * ML * 2;
    const double* R = right + (size_t)b * MR * 2;
    for (int e = lane; e < nl * nr; e += 32) {
        const int i = e / nr, j = e - i * nr;
        s_cost[i * MR + j] = okp_epipolar_cost(F, L[2 * i], L[2 * i + 1], R[2 * j], R[2 * j + 1]);
    }
    for (int i = lane; i < ML; i += 32) {
        match[(size_t)b * ML + i] = -1;
        match_cost[(size_t)b * ML + i] = 0.0;
    }
    if (lane == 0) { s_used_left = 0ull; s_used_right = 0ull; }
    __syncwarp();
    okp_greedy_match(s_cost, MR, nl, nr, max_distance, s_used_left, s_used_right, lane, [&](int i, int j, double cost) {
        match[(size_t)b * ML + i] = j;
        match_cost[(size_t)b * ML + i] = cost;
    });
}

// ---------------------------------------------------------------------------------------------
// Stereo objects: triangulate the decoded objects of P frame pairs (left frame, right frame) of one
// rig, one warp per pair. Statement of record: oracle/stereo_oracle.py::stereo_objects.
//   1. undistort every valid keypoint of both frames with its view's camera (lanes own keypoints);
//   2. match objects by their centre keypoints: okp_epipolar_cost + okp_greedy_match, as
//      okp_associate_kernel does (lanes own (left, right) cost entries);
//   3. for each matched object pair and spoke type, match the two objects' slots the same way;
//   4. triangulate every matched keypoint pair (lanes own pairs) like StereoCamera.triangulate: the
//      undistorted points rounded to float32, optionally okp_correct_pair (rounded to float32), then
//      the two-view DLT with P_L = K_L [I|0], P_R = K_R T_RL[:3], dehomogenised.
// Matching reads the unrounded undistorted points, as AssociationComponent does.
// Keypoints of an object are kept in compact order k = off[c] + s (P = 1 + sum(keypoint_config) of them).
// ---------------------------------------------------------------------------------------------
#include "okp_geometry.cuh"
#include "okp_dlt.cuh"

struct OkpStereoRig {
    OkpCamera cam[2];          // left, right
    OkpMat3 F;                 // x_R^T F x_L = 0
    OkpEpipoles ep;            // okp_epipoles(F), once per call on the host
    double proj[2][12];        // P_L, P_R row-major 3x4
};

struct OkpStereoShape {
    int N, C, O, S, P;         // P: keypoints per object (compact)
    int32_t cfg[OKP_MAX_MAPS]; // cfg[0] = 1
    int32_t off[OKP_MAX_MAPS]; // compact offset of map c
};

// Shared bytes per pair (one warp per CTA): undistorted points of both frames, centre costs, slot costs, matched-pair
// list, right slot of every left keypoint, matched right object of every left object, keypoint counts of both frames.
__host__ __device__ inline size_t okp_stereo_smem_bytes(int O, int C, int P) {
    return sizeof(double) * 2 * 2 * (size_t)O * P + sizeof(double) * (size_t)O * O + sizeof(double) * OKP_MAX_SLOTS * OKP_MAX_SLOTS +
           sizeof(uint32_t) * (size_t)O * P + (size_t)O * P + (size_t)O + 2 * (size_t)O * C;
}

__global__ void __launch_bounds__(32)
okp_stereo_objects_kernel(OkpStereoRig rig, OkpStereoShape d, const int32_t* __restrict__ n_objects,
                          const int32_t* __restrict__ kp_count, const float* __restrict__ kp_xy,
                          const int32_t* __restrict__ pairs, double max_distance, int optimal_correction,
                          OkpStereoTables out) {
    extern __shared__ double s_xy[];                              // [2][O][P][2]
    double* s_cost = s_xy + 4 * d.O * d.P;                        // [O][O] centre costs
    double* s_slot_cost = s_cost + d.O * d.O;                     // [8][8] slot costs of one (object pair, type)
    uint32_t* s_list = (uint32_t*)(s_slot_cost + OKP_MAX_SLOTS * OKP_MAX_SLOTS);   // matched keypoint pairs
    int8_t* s_slot = (int8_t*)(s_list + d.O * d.P);               // [O][P] right slot of a left keypoint, -1
    int8_t* s_object = s_slot + d.O * d.P;                        // [O] right object of a left object, -1
    int8_t* s_count = s_object + d.O;                             // [2][O][C] keypoints kept
    __shared__ unsigned long long s_used_left, s_used_right;
    __shared__ int s_n_list;
    const int p = blockIdx.x, lane = threadIdx.x;
    const int O = d.O, C = d.C, S = d.S, P = d.P;
    const int fl = pairs[2 * p], fr = pairs[2 * p + 1];
    const bool bad = fl < 0 || fl >= d.N || fr < 0 || fr >= d.N;
    const int nl = bad ? 0 : okp_clamp(n_objects[fl], 0, O), nr = bad ? 0 : okp_clamp(n_objects[fr], 0, O);
    for (int e = lane; e < 2 * O * C; e += 32) {
        const bool right = e >= O * C;
        const int o = (e / C) % O, c = e % C;
        s_count[e] = (int8_t)(o < (right ? nr : nl) ? okp_clamp(kp_count[((size_t)(right ? fr : fl) * O + o) * C + c], 0, d.cfg[c]) : 0);
    }
    for (int e = lane; e < O * P; e += 32) s_slot[e] = -1;
    for (int o = lane; o < O; o += 32) {
        s_object[o] = -1;
        out.object_match[(size_t)p * O + o] = -1;
        out.object_cost[(size_t)p * O + o] = 0.0;
    }
    if (lane == 0) { s_used_left = 0ull; s_used_right = 0ull; s_n_list = 0; }
    __syncwarp();
    // 1. undistortion
#pragma unroll
    for (int v = 0; v < 2; ++v) {
        const int f = v ? fr : fl;
        for (int e = lane; e < (v ? nr : nl) * C * S; e += 32) {
            const int o = e / (C * S), c = (e / S) % C, s = e % S;
            if (s >= s_count[(v * O + o) * C + c]) continue;
            const float* xy = kp_xy + ((((size_t)f * O + o) * C + c) * S + s) * 2;
            double* u = s_xy + 2 * ((v * O + o) * P + d.off[c] + s);
            okp_undistort_point((double)xy[0], (double)xy[1], rig.cam[v], u, u + 1);
        }
    }
    __syncwarp();
    // 2. objects by their centres
    const double* L = s_xy;
    const double* R = s_xy + 2 * O * P;
    for (int e = lane; e < nl * nr; e += 32) {
        const int i = e / nr, j = e - i * nr;
        s_cost[i * O + j] = okp_epipolar_cost(rig.F.m, L[2 * i * P], L[2 * i * P + 1], R[2 * j * P], R[2 * j * P + 1]);
    }
    __syncwarp();
    bool ambiguous = false;                                       // two or more right centres within reach of one left centre
    for (int i = lane; i < nl; i += 32) {
        int within = 0;
        for (int j = 0; j < nr; ++j) within += s_cost[i * O + j] <= max_distance;
        ambiguous |= within >= 2;
    }
    ambiguous = __any_sync(0xffffffffu, ambiguous);
    okp_greedy_match(s_cost, O, nl, nr, max_distance, s_used_left, s_used_right, lane, [&](int i, int j, double cost) {
        out.object_match[(size_t)p * O + i] = j;
        out.object_cost[(size_t)p * O + i] = cost;
        s_object[i] = (int8_t)j;
        s_slot[i * P] = 0;
        s_list[s_n_list++] = (uint32_t)i | (uint32_t)j << 8;      // left object, right object, map 0, slots 0
    });
    __syncwarp();
    // 3. slots of every matched object pair, type by type
    for (int i = 0; i < nl; ++i) {
        const int j = s_object[i];
        if (j < 0) continue;
        for (int c = 1; c < C; ++c) {
            const int nsl = s_count[i * C + c], nsr = s_count[(O + j) * C + c];
            if (nsl == 0 || nsr == 0) continue;
            const double* Ls = L + 2 * (i * P + d.off[c]);
            const double* Rs = R + 2 * (j * P + d.off[c]);
            for (int e = lane; e < nsl * nsr; e += 32) {
                const int a = e / nsr, b = e - a * nsr;
                s_slot_cost[a * OKP_MAX_SLOTS + b] = okp_epipolar_cost(rig.F.m, Ls[2 * a], Ls[2 * a + 1], Rs[2 * b], Rs[2 * b + 1]);
            }
            if (lane == 0) { s_used_left = 0ull; s_used_right = 0ull; }
            __syncwarp();
            okp_greedy_match(s_slot_cost, OKP_MAX_SLOTS, nsl, nsr, max_distance, s_used_left, s_used_right, lane,
                             [&](int a, int b, double) {
                s_slot[i * P + d.off[c] + a] = (int8_t)b;
                s_list[s_n_list++] = (uint32_t)i | (uint32_t)j << 8 | (uint32_t)c << 16 | (uint32_t)a << 20 | (uint32_t)b << 24;
            });
            __syncwarp();
        }
    }
    // slot_match for every slot; NaN points where nothing is matched
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    for (int e = lane; e < O * C * S; e += 32) {
        const int o = e / (C * S), c = (e / S) % C, s = e % S;
        const int m = s < d.cfg[c] ? s_slot[o * P + d.off[c] + s] : -1;
        const size_t at = (size_t)p * O * C * S + e;
        out.slot_match[at] = m;
        if (m < 0) { out.point[3 * at] = nan; out.point[3 * at + 1] = nan; out.point[3 * at + 2] = nan; }
    }
    // 4. correction + DLT of every matched keypoint pair
    for (int e = lane; e < s_n_list; e += 32) {
        const uint32_t w = s_list[e];
        const int i = w & 255, j = (w >> 8) & 255, c = (w >> 16) & 15, a = (w >> 20) & 15, b = w >> 24;
        const double* l = L + 2 * (i * P + d.off[c] + a);
        const double* r = R + 2 * (j * P + d.off[c] + b);
        double x[2][2] = {{(double)(float)l[0], (double)(float)l[1]}, {(double)(float)r[0], (double)(float)r[1]}};
        if (optimal_correction) {
            okp_correct_pair(rig.F, rig.ep, x[0][0], x[0][1], x[1][0], x[1][1], x[0], x[1]);
#pragma unroll
            for (int v = 0; v < 2; ++v) { x[v][0] = (double)(float)x[v][0]; x[v][1] = (double)(float)x[v][1]; }
        }
        double A[4][4] = {};
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            const double* M = rig.proj[v];
            double row[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) row[k] = x[v][0] * M[8 + k] - M[k];
            okp_givens_append(A, row);
#pragma unroll
            for (int k = 0; k < 4; ++k) row[k] = x[v][1] * M[8 + k] - M[4 + k];
            okp_givens_append(A, row);
        }
        double h[4];
        okp_smallest_right_singular_vector(A, h);
        double* X = out.point + 3 * ((((size_t)p * O + i) * C + c) * S + a);
        X[0] = h[0] / h[3]; X[1] = h[1] / h[3]; X[2] = h[2] / h[3];
    }
    if (lane == 0) out.flags[p] = (bad ? OKP_STEREO_BAD_PAIR : 0u) | (ambiguous ? OKP_STEREO_AMBIGUOUS : 0u);
}

// ---------------------------------------------------------------------------------------------
// Stereo objects, depth association (okp_triangulate_stereo_objects_depth_f64): the steps of okp_stereo_objects_kernel,
// with every candidate scored by where each view's monocular lift (kp_point, in its own camera's frame) lands in the
// other view. Statement of record: oracle/stereo_depth_oracle.py::stereo_objects_depth.
//   1. every valid keypoint is undistorted (u) and its lift X projected into the other view, q = pi(K (R X + t)) with
//      that view's fx, fy, cx, cy (NaN unless X is finite with z > 0): q_R of a left keypoint, q_L of a right one;
//   2./3. candidate (i, j) is admissible when okp_epipolar_cost(u_L(i), u_R(j)) <= max_distance and
//      d(i, j) <= max_depth, d = 0.5 (|q_R(i) - u_R(j)| + |q_L(j) - u_L(i)|), or the one term whose lift exists;
//      okp_greedy_match runs on d (INFINITY where the epipolar gate fails), centres first, then slots type by type. A
//      candidate inside the epipolar gate with no lift on either side is never matched and sets OKP_STEREO_NO_DEPTH;
//      OKP_STEREO_AMBIGUOUS marks a left object with two or more admissible right objects;
//   4. unchanged: correction + DLT of every matched keypoint pair, object_cost holds d.
// This kernel repeats okp_stereo_objects_kernel's structure instead of sharing one inline body with it: that kernel's
// body is left untouched, so its SASS stays what it was.
// ---------------------------------------------------------------------------------------------
struct OkpStereoLift {
    double R[2][9];            // [0]: R_RL (a left lift into the right camera), [1]: R_LR = R_RL^T; row-major
    double t[2][3];            // [0]: t_RL, [1]: t_LR = -R_RL^T t_RL
};

// okp_stereo_smem_bytes plus the projected lifts q of both frames, [2][O][P][2] doubles after the undistorted points
__host__ __device__ inline size_t okp_stereo_depth_smem_bytes(int O, int C, int P) {
    return okp_stereo_smem_bytes(O, C, P) + sizeof(double) * 2 * 2 * (size_t)O * P;
}

// q = pi(K (R X + t)) in the undistorted pixels of `cam`; NaN unless the lift is finite with z > 0
__device__ __forceinline__ void okp_project_lift(const double* X, const double* R, const double* t, const OkpCamera& cam,
                                                 double* q) {
    const double x = X[0], y = X[1], z = X[2];
    if (!(isfinite(x) && isfinite(y) && isfinite(z) && z > 0.0)) {
        q[0] = q[1] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    const double Y0 = R[0] * x + R[1] * y + R[2] * z + t[0];
    const double Y1 = R[3] * x + R[4] * y + R[5] * z + t[1];
    const double Y2 = R[6] * x + R[7] * y + R[8] * z + t[2];
    q[0] = (cam.fx * Y0 + cam.cx * Y2) / Y2;
    q[1] = (cam.fy * Y1 + cam.cy * Y2) / Y2;
}

// The cost of candidate (left keypoint: u_L, q_R; right keypoint: u_R, q_L): d when it passes the epipolar gate,
// INFINITY otherwise; sets no_depth for a candidate inside the gate whose lifts are both missing.
__device__ __forceinline__ double okp_depth_cost(const double* F, const double* uL, const double* qR, const double* uR,
                                                 const double* qL, double max_distance, bool& no_depth) {
    if (!(okp_epipolar_cost(F, uL[0], uL[1], uR[0], uR[1]) <= max_distance)) return INFINITY;
    const bool has_r = qR[0] == qR[0], has_l = qL[0] == qL[0];
    if (!has_r && !has_l) { no_depth = true; return INFINITY; }
    double a = 0.0, b = 0.0;
    if (has_r) { const double dx = qR[0] - uR[0], dy = qR[1] - uR[1]; a = sqrt(dx * dx + dy * dy); }
    if (has_l) { const double dx = qL[0] - uL[0], dy = qL[1] - uL[1]; b = sqrt(dx * dx + dy * dy); }
    return has_r && has_l ? 0.5 * (a + b) : (has_r ? a : b);
}

__global__ void __launch_bounds__(32)
okp_stereo_depth_kernel(OkpStereoRig rig, OkpStereoLift lift, OkpStereoShape d, const int32_t* __restrict__ n_objects,
                        const int32_t* __restrict__ kp_count, const float* __restrict__ kp_xy,
                        const double* __restrict__ kp_point, const int32_t* __restrict__ pairs, double max_distance,
                        double max_depth, int optimal_correction, OkpStereoTables out) {
    extern __shared__ double s_xy[];                              // [2][O][P][2] undistorted points u
    double* s_q = s_xy + 4 * d.O * d.P;                           // [2][O][P][2] lifts projected into the other view
    double* s_cost = s_q + 4 * d.O * d.P;                         // [O][O] centre costs
    double* s_slot_cost = s_cost + d.O * d.O;                     // [8][8] slot costs of one (object pair, type)
    uint32_t* s_list = (uint32_t*)(s_slot_cost + OKP_MAX_SLOTS * OKP_MAX_SLOTS);   // matched keypoint pairs
    int8_t* s_slot = (int8_t*)(s_list + d.O * d.P);               // [O][P] right slot of a left keypoint, -1
    int8_t* s_object = s_slot + d.O * d.P;                        // [O] right object of a left object, -1
    int8_t* s_count = s_object + d.O;                             // [2][O][C] keypoints kept
    __shared__ unsigned long long s_used_left, s_used_right;
    __shared__ int s_n_list;
    const int p = blockIdx.x, lane = threadIdx.x;
    const int O = d.O, C = d.C, S = d.S, P = d.P;
    const int fl = pairs[2 * p], fr = pairs[2 * p + 1];
    const bool bad = fl < 0 || fl >= d.N || fr < 0 || fr >= d.N;
    const int nl = bad ? 0 : okp_clamp(n_objects[fl], 0, O), nr = bad ? 0 : okp_clamp(n_objects[fr], 0, O);
    for (int e = lane; e < 2 * O * C; e += 32) {
        const bool right = e >= O * C;
        const int o = (e / C) % O, c = e % C;
        s_count[e] = (int8_t)(o < (right ? nr : nl) ? okp_clamp(kp_count[((size_t)(right ? fr : fl) * O + o) * C + c], 0, d.cfg[c]) : 0);
    }
    for (int e = lane; e < O * P; e += 32) s_slot[e] = -1;
    for (int o = lane; o < O; o += 32) {
        s_object[o] = -1;
        out.object_match[(size_t)p * O + o] = -1;
        out.object_cost[(size_t)p * O + o] = 0.0;
    }
    if (lane == 0) { s_used_left = 0ull; s_used_right = 0ull; s_n_list = 0; }
    __syncwarp();
    // 1. undistortion, and every lift projected into the other view
#pragma unroll
    for (int v = 0; v < 2; ++v) {
        const int f = v ? fr : fl;
        for (int e = lane; e < (v ? nr : nl) * C * S; e += 32) {
            const int o = e / (C * S), c = (e / S) % C, s = e % S;
            if (s >= s_count[(v * O + o) * C + c]) continue;
            const size_t at = (((size_t)f * O + o) * C + c) * S + s;
            const int k = 2 * ((v * O + o) * P + d.off[c] + s);
            okp_undistort_point((double)kp_xy[2 * at], (double)kp_xy[2 * at + 1], rig.cam[v], s_xy + k, s_xy + k + 1);
            okp_project_lift(kp_point + 3 * at, lift.R[v], lift.t[v], rig.cam[1 - v], s_q + k);
        }
    }
    __syncwarp();
    // 2. objects by their centres
    const double* L = s_xy;
    const double* R = s_xy + 2 * O * P;
    const double* QR = s_q;                                       // left keypoints' lifts in the right view
    const double* QL = s_q + 2 * O * P;                           // right keypoints' lifts in the left view
    bool no_depth = false;
    for (int e = lane; e < nl * nr; e += 32) {
        const int i = e / nr, j = e - i * nr;
        s_cost[i * O + j] = okp_depth_cost(rig.F.m, L + 2 * i * P, QR + 2 * i * P, R + 2 * j * P, QL + 2 * j * P, max_distance,
                                           no_depth);
    }
    __syncwarp();
    bool ambiguous = false;                                       // two or more admissible right objects of one left object
    for (int i = lane; i < nl; i += 32) {
        int within = 0;
        for (int j = 0; j < nr; ++j) within += s_cost[i * O + j] <= max_depth;
        ambiguous |= within >= 2;
    }
    ambiguous = __any_sync(0xffffffffu, ambiguous);
    okp_greedy_match(s_cost, O, nl, nr, max_depth, s_used_left, s_used_right, lane, [&](int i, int j, double cost) {
        out.object_match[(size_t)p * O + i] = j;
        out.object_cost[(size_t)p * O + i] = cost;
        s_object[i] = (int8_t)j;
        s_slot[i * P] = 0;
        s_list[s_n_list++] = (uint32_t)i | (uint32_t)j << 8;      // left object, right object, map 0, slots 0
    });
    __syncwarp();
    // 3. slots of every matched object pair, type by type
    for (int i = 0; i < nl; ++i) {
        const int j = s_object[i];
        if (j < 0) continue;
        for (int c = 1; c < C; ++c) {
            const int nsl = s_count[i * C + c], nsr = s_count[(O + j) * C + c];
            if (nsl == 0 || nsr == 0) continue;
            const int kl = 2 * (i * P + d.off[c]), kr = 2 * (j * P + d.off[c]);
            for (int e = lane; e < nsl * nsr; e += 32) {
                const int a = e / nsr, b = e - a * nsr;
                s_slot_cost[a * OKP_MAX_SLOTS + b] = okp_depth_cost(rig.F.m, L + kl + 2 * a, QR + kl + 2 * a, R + kr + 2 * b,
                                                                    QL + kr + 2 * b, max_distance, no_depth);
            }
            if (lane == 0) { s_used_left = 0ull; s_used_right = 0ull; }
            __syncwarp();
            okp_greedy_match(s_slot_cost, OKP_MAX_SLOTS, nsl, nsr, max_depth, s_used_left, s_used_right, lane,
                             [&](int a, int b, double) {
                s_slot[i * P + d.off[c] + a] = (int8_t)b;
                s_list[s_n_list++] = (uint32_t)i | (uint32_t)j << 8 | (uint32_t)c << 16 | (uint32_t)a << 20 | (uint32_t)b << 24;
            });
            __syncwarp();
        }
    }
    no_depth = __any_sync(0xffffffffu, no_depth);
    // slot_match for every slot; NaN points where nothing is matched
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    for (int e = lane; e < O * C * S; e += 32) {
        const int o = e / (C * S), c = (e / S) % C, s = e % S;
        const int m = s < d.cfg[c] ? s_slot[o * P + d.off[c] + s] : -1;
        const size_t at = (size_t)p * O * C * S + e;
        out.slot_match[at] = m;
        if (m < 0) { out.point[3 * at] = nan; out.point[3 * at + 1] = nan; out.point[3 * at + 2] = nan; }
    }
    // 4. correction + DLT of every matched keypoint pair
    for (int e = lane; e < s_n_list; e += 32) {
        const uint32_t w = s_list[e];
        const int i = w & 255, j = (w >> 8) & 255, c = (w >> 16) & 15, a = (w >> 20) & 15, b = w >> 24;
        const double* l = L + 2 * (i * P + d.off[c] + a);
        const double* r = R + 2 * (j * P + d.off[c] + b);
        double x[2][2] = {{(double)(float)l[0], (double)(float)l[1]}, {(double)(float)r[0], (double)(float)r[1]}};
        if (optimal_correction) {
            okp_correct_pair(rig.F, rig.ep, x[0][0], x[0][1], x[1][0], x[1][1], x[0], x[1]);
#pragma unroll
            for (int v = 0; v < 2; ++v) { x[v][0] = (double)(float)x[v][0]; x[v][1] = (double)(float)x[v][1]; }
        }
        double A[4][4] = {};
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            const double* M = rig.proj[v];
            double row[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) row[k] = x[v][0] * M[8 + k] - M[k];
            okp_givens_append(A, row);
#pragma unroll
            for (int k = 0; k < 4; ++k) row[k] = x[v][1] * M[8 + k] - M[4 + k];
            okp_givens_append(A, row);
        }
        double h[4];
        okp_smallest_right_singular_vector(A, h);
        double* X = out.point + 3 * ((((size_t)p * O + i) * C + c) * S + a);
        X[0] = h[0] / h[3]; X[1] = h[1] / h[3]; X[2] = h[2] / h[3];
    }
    if (lane == 0)
        out.flags[p] = (bad ? OKP_STEREO_BAD_PAIR : 0u) | (ambiguous ? OKP_STEREO_AMBIGUOUS : 0u) |
                       (no_depth ? OKP_STEREO_NO_DEPTH : 0u);
}
