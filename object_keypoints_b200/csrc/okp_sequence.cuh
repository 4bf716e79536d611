// okp_sequence.cuh -- the decoded objects of a posed sequence, matched from every anchor frame into its V - 1 view frames
// (okp_triangulate_sequence_objects_f64). Statement of record: oracle/sequence_objects_oracle.py::sequence_objects.
//
// okp_sequence_match_kernel runs one warp per (anchor a, view v >= 1) pair, in the structure of okp_stereo_depth_kernel
// with the anchor frame frames[a, 0] as the left view and frames[a, v] as the right one. Both come from one camera, and
// the pair's geometry is read from device arrays indexed by the pair instead of host scalars:
//   1. every valid keypoint of both frames is undistorted; with association 1 its lift (kp_point) is projected into the
//      other frame with the pair's rigid motion (anchor -> view) or its inverse;
//   2./3. objects are matched by their centres, then each matched pair's slots type by type, with okp_greedy_match on
//      association 0: okp_epipolar_cost under the pair's F, while <= max_distance (okp_stereo_objects_kernel's rule);
//      association 1: okp_depth_cost, the epipolar gate then d <= max_depth (okp_stereo_depth_kernel's rule, with its
//      OKP_STEREO_NO_DEPTH and OKP_STEREO_AMBIGUOUS semantics);
//   4. the match tables, and the tracks of every anchor slot: column v of observations / observed / valid holds the
//      matched view keypoint (distorted pixels, kp_xy) or nothing; the v = 1 warp also writes column 0, the anchor's own
//      keypoint. error is set to NaN here: the track kernel overwrites it for every track with two or more views.
// okp_triangulate_robust_kernel then solves the tracks, one group per anchor, unchanged.
#pragma once
#include "okp_stereo.cuh"

// Shared bytes per pair: undistorted points u and projected lifts q of both frames ([2][O][P][2] doubles each), centre
// costs [O][O], slot costs [8][8], the view slot of every anchor keypoint [O][P], the view object of every anchor object
// [O], keypoint counts of both frames [2][O][C]. okp_stereo_depth_smem_bytes without its list of matched keypoint pairs:
// nothing is triangulated in this kernel.
__host__ __device__ inline size_t okp_sequence_smem_bytes(int O, int C, int P) {
    return sizeof(double) * (8 * (size_t)O * P + (size_t)O * O + OKP_MAX_SLOTS * OKP_MAX_SLOTS) + (size_t)O * P + (size_t)O +
           2 * (size_t)O * C;
}

__global__ void __launch_bounds__(32)
okp_sequence_match_kernel(OkpCamera cam, OkpStereoShape d, int V, const int32_t* __restrict__ n_objects,
                          const int32_t* __restrict__ kp_count, const float* __restrict__ kp_xy,
                          const double* __restrict__ kp_point, const int32_t* __restrict__ frames,
                          const double* __restrict__ F_pairs, const double* __restrict__ motion, int association,
                          double max_distance, double max_depth, OkpSequenceObjectTables out) {
    extern __shared__ double s_xy[];                              // [2][O][P][2] undistorted points u: anchor, view
    double* s_q = s_xy + 4 * d.O * d.P;                           // [2][O][P][2] lifts projected into the other frame
    double* s_cost = s_q + 4 * d.O * d.P;                         // [O][O] centre costs
    double* s_slot_cost = s_cost + d.O * d.O;                     // [8][8] slot costs of one (object pair, type)
    int8_t* s_slot = (int8_t*)(s_slot_cost + OKP_MAX_SLOTS * OKP_MAX_SLOTS);   // [O][P] view slot of an anchor keypoint
    int8_t* s_object = s_slot + d.O * d.P;                        // [O] view object of an anchor object, -1
    int8_t* s_count = s_object + d.O;                             // [2][O][C] keypoints kept
    __shared__ unsigned long long s_used_left, s_used_right;
    const int pair = blockIdx.x, lane = threadIdx.x;              // pair = a (V - 1) + v - 1
    const int a = pair / (V - 1), v = pair - a * (V - 1) + 1;
    const int O = d.O, C = d.C, S = d.S, P = d.P;
    const bool depth = association != 0;
    const int fl = frames[(size_t)a * V], fr = frames[(size_t)a * V + v];
    const bool anchor_ok = fl >= 0 && fl < d.N, view_ok = fr >= 0 && fr < d.N, bad = !anchor_ok || !view_ok;
    const int na = anchor_ok ? okp_clamp(n_objects[fl], 0, O) : 0;   // the anchor's objects: column 0 of its tracks
    const int nl = bad ? 0 : na, nr = bad ? 0 : okp_clamp(n_objects[fr], 0, O);
    const double* F = F_pairs + 9 * (size_t)pair;
    const double* Rt = depth ? motion + 24 * (size_t)pair : nullptr;   // [2][12]: R row-major, t; [0] anchor -> view
    const double gate = depth ? max_depth : max_distance;
    for (int e = lane; e < 2 * O * C; e += 32) {
        const bool right = e >= O * C;
        const int o = (e / C) % O, c = e % C;
        s_count[e] = (int8_t)(o < (right ? nr : na) ? okp_clamp(kp_count[((size_t)(right ? fr : fl) * O + o) * C + c], 0, d.cfg[c]) : 0);
    }
    for (int e = lane; e < O * P; e += 32) s_slot[e] = -1;
    for (int o = lane; o < O; o += 32) {
        s_object[o] = -1;
        out.object_match[(size_t)pair * O + o] = -1;
        out.object_cost[(size_t)pair * O + o] = 0.0;
    }
    if (lane == 0) { s_used_left = 0ull; s_used_right = 0ull; }
    __syncwarp();
    // 1. undistortion, and (depth) every lift projected into the other frame
#pragma unroll
    for (int w = 0; w < 2; ++w) {
        const int f = w ? fr : fl;
        for (int e = lane; e < (w ? nr : nl) * C * S; e += 32) {
            const int o = e / (C * S), c = (e / S) % C, s = e % S;
            if (s >= s_count[(w * O + o) * C + c]) continue;
            const size_t at = (((size_t)f * O + o) * C + c) * S + s;
            const int k = 2 * ((w * O + o) * P + d.off[c] + s);
            okp_undistort_point((double)kp_xy[2 * at], (double)kp_xy[2 * at + 1], cam, s_xy + k, s_xy + k + 1);
            if (depth) okp_project_lift(kp_point + 3 * at, Rt + 12 * w, Rt + 12 * w + 9, cam, s_q + k);
        }
    }
    __syncwarp();
    // 2. objects by their centres
    const double* L = s_xy;
    const double* R = s_xy + 2 * O * P;
    const double* QR = s_q;                                       // anchor keypoints' lifts in the view frame
    const double* QL = s_q + 2 * O * P;                           // view keypoints' lifts in the anchor frame
    bool no_depth = false;
    for (int e = lane; e < nl * nr; e += 32) {
        const int i = e / nr, j = e - i * nr;
        const int kl = 2 * i * P, kr = 2 * j * P;
        s_cost[i * O + j] = depth ? okp_depth_cost(F, L + kl, QR + kl, R + kr, QL + kr, max_distance, no_depth)
                                  : okp_epipolar_cost(F, L[kl], L[kl + 1], R[kr], R[kr + 1]);
    }
    __syncwarp();
    bool ambiguous = false;                                       // two or more admissible view objects of one anchor object
    for (int i = lane; i < nl; i += 32) {
        int within = 0;
        for (int j = 0; j < nr; ++j) within += s_cost[i * O + j] <= gate;
        ambiguous |= within >= 2;
    }
    ambiguous = __any_sync(0xffffffffu, ambiguous);
    okp_greedy_match(s_cost, O, nl, nr, gate, s_used_left, s_used_right, lane, [&](int i, int j, double cost) {
        out.object_match[(size_t)pair * O + i] = j;
        out.object_cost[(size_t)pair * O + i] = cost;
        s_object[i] = (int8_t)j;
        s_slot[i * P] = 0;
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
                const int sa = e / nsr, sb = e - sa * nsr;
                const int l = kl + 2 * sa, r = kr + 2 * sb;
                s_slot_cost[sa * OKP_MAX_SLOTS + sb] = depth ? okp_depth_cost(F, L + l, QR + l, R + r, QL + r, max_distance, no_depth)
                                                             : okp_epipolar_cost(F, L[l], L[l + 1], R[r], R[r + 1]);
            }
            if (lane == 0) { s_used_left = 0ull; s_used_right = 0ull; }
            __syncwarp();
            okp_greedy_match(s_slot_cost, OKP_MAX_SLOTS, nsl, nsr, gate, s_used_left, s_used_right, lane,
                             [&](int sa, int sb, double) { s_slot[i * P + d.off[c] + sa] = (int8_t)sb; });
            __syncwarp();
        }
    }
    no_depth = __any_sync(0xffffffffu, no_depth);
    // 4. slot_match, and column v (the v = 1 warp: column 0 too) of every anchor slot's track
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    for (int e = lane; e < O * C * S; e += 32) {
        const int o = e / (C * S), c = (e / S) % C, s = e % S;
        const int m = s < d.cfg[c] ? s_slot[o * P + d.off[c] + s] : -1;
        out.slot_match[(size_t)pair * O * C * S + e] = m;
        const size_t track = (size_t)a * O * C * S + e;           // [A][O][C][S] tracks of V views
        double x = 0.0, y = 0.0;
        if (m >= 0) {
            const size_t at = (((size_t)fr * O + s_object[o]) * C + c) * S + m;
            x = (double)kp_xy[2 * at]; y = (double)kp_xy[2 * at + 1];
        }
        size_t tv = track * V + v;
        out.observations[2 * tv] = x; out.observations[2 * tv + 1] = y;
        out.observed[tv] = out.valid[tv] = (uint8_t)(m >= 0);
        out.error[tv] = nan;
        if (v == 1) {
            const bool own = s < s_count[o * C + c];
            x = y = 0.0;
            if (own) {
                const size_t at = (((size_t)fl * O + o) * C + c) * S + s;
                x = (double)kp_xy[2 * at]; y = (double)kp_xy[2 * at + 1];
            }
            tv = track * V;
            out.observations[2 * tv] = x; out.observations[2 * tv + 1] = y;
            out.observed[tv] = out.valid[tv] = (uint8_t)own;
            out.error[tv] = nan;
        }
    }
    if (lane == 0)
        out.flags[pair] = (bad ? OKP_STEREO_BAD_PAIR : 0u) | (ambiguous ? OKP_STEREO_AMBIGUOUS : 0u) |
                          (no_depth ? OKP_STEREO_NO_DEPTH : 0u);
}
