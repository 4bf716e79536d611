// okp_group.cuh -- K3 + K4: centre-vector voting into object instances, over-detection
// resolution and 3D points. One WARP per frame; everything it touches is a few hundred bytes of
// peak records plus 3 gathered floats per spoke peak (2 centre-vector components, 1 depth).
//
// Replaces ObjectExtraction.__call__ (perception/pipeline.py:104-153) and the DetectionToPoint
// loop of ObjectKeypointPipeline.__call__ (pipeline.py:189-199).
//
// okp_group_frame() is the one statement of that arithmetic. It runs in two places:
//   * in the epilogue warps of the fused decode kernel (okp_peaks_stream.cuh, FUSED = true), straight from the
//     frame's sorted peak list in shared memory while the compute warps stream the next frames -- the normal path;
//   * in okp_group_kernel below, which first pulls the frame's peak tables from HBM: the stand-alone entry
//     (okp_group_objects_*), shapes the fused kernel does not cover, and the fix-up of frames one of whose maps
//     took the overflow path (marked by n_objects = OKP_GROUP_PENDING);
//   * in okp_group_cameras_kernel, the same steps with one camera per frame (okp_*_cameras_*).
#pragma once
#include "okp_common.cuh"
#include "okp_geometry.cuh"
#include "okp_records.cuh"

#define OKP_KMEANS_MAX_INITS 256


// Deterministic stand-in for the reference's unseeded KMeans(init='random') (pipeline.py:146-148):
// Lloyd's algorithm from every k-subset of the detections (lexicographic, at most
// OKP_KMEANS_MAX_INITS), lowest inertia wins. Same statement as oracle/okp_oracle.c.
// xy: the map's peak_xy table; idx[0..n): the detections of this (object, type). Points are re-read
// from the table instead of being copied, to keep the per-thread stack small.
__device__ __noinline__ void okp_cluster_detections(const float* __restrict__ xy, const unsigned char* idx, int n, int k,
                                                    int iters, float* out) {
#define OKP_PT(i, d) ((double)xy[2 * (int)idx[(i)] + (d)])
    double cen[OKP_MAX_SLOTS][2], best_cen[OKP_MAX_SLOTS][2];
    int subset[OKP_MAX_SLOTS];
    unsigned char assign[OKP_MAX_PEAKS], new_assign[OKP_MAX_PEAKS];
    double best = 0.0;
    bool have_best = false;
    for (int c = 0; c < k; ++c) subset[c] = c;
    for (int init = 0; init < OKP_KMEANS_MAX_INITS; ++init) {
        for (int c = 0; c < k; ++c) { cen[c][0] = OKP_PT(subset[c], 0); cen[c][1] = OKP_PT(subset[c], 1); }
        bool have_assign = false;
        for (int it = 0; it < iters; ++it) {
            bool same = have_assign;
            for (int i = 0; i < n; ++i) {
                int arg = 0;
                double dmin = 0.0;
                for (int c = 0; c < k; ++c) {
                    const double dx = OKP_PT(i, 0) - cen[c][0], dy = OKP_PT(i, 1) - cen[c][1];
                    const double d = dx * dx + dy * dy;
                    if (c == 0 || d < dmin) { dmin = d; arg = c; }
                }
                new_assign[i] = (unsigned char)arg;
                if (have_assign && assign[i] != arg) same = false;
            }
            if (same) break;
            for (int i = 0; i < n; ++i) assign[i] = new_assign[i];
            have_assign = true;
            for (int c = 0; c < k; ++c) {
                double sx = 0.0, sy = 0.0;
                int m = 0;
                for (int i = 0; i < n; ++i)
                    if (assign[i] == c) { sx += OKP_PT(i, 0); sy += OKP_PT(i, 1); ++m; }
                if (m) { cen[c][0] = sx / m; cen[c][1] = sy / m; }
            }
        }
        double inertia = 0.0;
        for (int i = 0; i < n; ++i) {
            double dmin = 0.0;
            for (int c = 0; c < k; ++c) {
                const double dx = OKP_PT(i, 0) - cen[c][0], dy = OKP_PT(i, 1) - cen[c][1];
                const double d = dx * dx + dy * dy;
                if (c == 0 || d < dmin) dmin = d;
            }
            inertia += dmin;
        }
        if (!have_best || inertia < best) {
            best = inertia;
            have_best = true;
            for (int c = 0; c < k; ++c) { best_cen[c][0] = cen[c][0]; best_cen[c][1] = cen[c][1]; }
        }
        int c = k - 1;
        while (c >= 0 && subset[c] == n - k + c) --c;
        if (c < 0) break;
        ++subset[c];
        for (int j = c + 1; j < k; ++j) subset[j] = subset[j - 1] + 1;
    }
    for (int c = 0; c < k; ++c) { out[2 * c] = (float)best_cen[c][0]; out[2 * c + 1] = (float)best_cen[c][1]; }
#undef OKP_PT
}


#define OKP_GROUP_PENDING (-1)      // n_objects marker: the frame's grouping is left to the fix-up launch

// What the grouping needs besides the peak list (one kernel parameter, read from the constant bank).
struct OkpGroupArgs {
    const void* depth;              // [N,C,H,W]     element type E (device memory or a pinned-host alias: gather-only)
    const void* centers;            // [N,C-1,2,H,W]
    OkpConfig config;
    OkpCamera cam;
    OkpDecodeParams prm;
    OkpRecordSinks sinks;           // optional compact records (okp_records.cuh); n = 0: none
    int N, C, H, W;
    int S;                          // max(1, max(keypoint_config))
    int P;                          // points per object in a record: 1 + sum(keypoint_config)
    int have_camera;
    int frame_smem_bytes;           // okp_group_smem_bytes()
};

// Shared-memory bytes ONE frame (= one warp) of the grouping needs. The per-frame-camera form (okp_group_cameras_kernel)
// keeps the frame's OkpCamera behind the scratch: the last sizeof(OkpCamera) bytes, 16-byte aligned.
static_assert(sizeof(OkpCamera) % 16 == 0, "OkpCamera is copied as 16-byte words");
static inline size_t okp_group_smem_bytes(int C, int K, int O, bool per_frame_camera = false) {
    size_t bytes = (size_t)O * 2 * sizeof(double);                                                  // centres
    bytes += (size_t)C * K * (2 * sizeof(double) + 2 * sizeof(float) + sizeof(float) + 2 * sizeof(int));
    bytes += (size_t)O * C * sizeof(int) + (size_t)O * sizeof(int);
    bytes += (2 * OKP_MAX_MAPS + 2) * sizeof(int);                                                  // counts, starts, flags
    return (bytes + 15) / 16 * 16 + (per_frame_camera ? sizeof(OkpCamera) : 0);
}

// The frame's scratch, carved out of `mine` (okp_group_smem_bytes() bytes, 16-byte aligned).
struct OkpGroupScratch {
    double (*center)[2];            // [O][2]
    double* vote;                   // [C][K][2] predicted centre of a spoke peak
    float* xy;                      // [C][K][2] centroid (x, y)        -- filled by the caller
    float* conf;                    // [C][K]                           -- filled by the caller
    int* obj;                       // [C][K]    object of a peak, -1 = none
    int* rank;                      // [C][K]    position of a spoke peak among the peaks of its (object, map)
    int* assigned;                  // [O][C]    detections per (object, map)
    int* nvotes;                    // [O]       votes per object
    int* counts;                    // [OKP_MAX_MAPS] min(peaks of the map, K) -- filled by the caller
    int* start;                     // [OKP_MAX_MAPS + 1] prefix of counts: the frame's peaks as one compact list
    unsigned int* flags;            // [1]       OKP_FLAG_* seen so far     -- initialised by the caller
};

__device__ __forceinline__ OkpGroupScratch okp_group_scratch(unsigned char* mine, int C, int K, int O) {
    OkpGroupScratch g;
    g.center = reinterpret_cast<double (*)[2]>(mine);
    g.vote = reinterpret_cast<double*>(mine) + (size_t)O * 2;
    g.xy = reinterpret_cast<float*>(g.vote + (size_t)C * K * 2);
    g.conf = g.xy + (size_t)C * K * 2;
    g.obj = reinterpret_cast<int*>(g.conf + (size_t)C * K);
    g.rank = g.obj + (size_t)C * K;
    g.assigned = g.rank + (size_t)C * K;
    g.nvotes = g.assigned + (size_t)O * C;
    g.counts = g.nvotes + O;
    g.start = g.counts + OKP_MAX_MAPS;
    g.flags = reinterpret_cast<unsigned int*>(g.start + OKP_MAX_MAPS + 1);
    return g;
}

// Grouping + 3D lift of ONE frame by ONE warp. Expects g.xy / g.conf / g.counts / g.flags to hold the frame's peaks
// (raster order per map).
//
// Shape of the work (round 2). A frame is ~10-40 peaks; the first version of this routine gave a lane to every
// (object), then every (object, map), then every (object, map, slot) and let it scan the peak lists -- ten active lanes
// per instruction and, measured in the fused kernel, more issue slots for the per-object vote lists than for the float64
// Newton iterations. Now the frame's peaks are ONE compact list (map-major, raster order inside a map = the order the
// reference walks them in, pipeline.py:115-128) and a lane owns a PEAK:
//   pass 1  spoke peaks: centre-vector gather, vote, nearest centre (squared distances; a square root only for the
//           minimum and for distances within rounding of it, which decides np.argmin's first-minimum rule exactly);
//           __match_any_sync over (object) and (object, map) gives every peak its slot in the object's vote list and
//           its rank among the detections of its (object, map) without any scan;
//   (o, c)  one lane per (object, map): counts, and the rare over-detection cases (arg-max confidence / clustering);
//   pass 2  every peak that is kept writes its keypoint slot and lifts itself to 3D (Newton undistortion + tan in
//           float64 -- two warp passes for 40 peaks instead of three over padded [O][C][S] slots).
// Global round trips on the critical path: centre-vector gather -> depth gather. No block-level barrier.
//   OkpDecodeParams.lean_tables == 0: every slot of the frame's object tables that is not written is reset (zero / -1),
//                  as include/okp.h promises by default;
//   lean_tables == 1: only the valid slots are written (the tables of a 64x64 frame are a quarter of its heatmap
//                  bytes; clearing them costs more DRAM traffic than the frame's peaks).
// LANES = 32: a warp per frame. LANES = 16: half a warp per frame (small frames -- a 64x64 valve frame is ~10 peaks, and
// the kernel is issue-bound with 12 active lanes per instruction: two frames per warp halve the warp instructions per
// frame). `lane` is the thread's index inside its frame, FULL the mask of the frame's lanes in the warp; the two halves of
// a warp run independently (every warp-level primitive below names the frame's own mask).
// FRAME_CAMERA = false: the frame is lifted with the call's camera a.cam; true: with *frame_camera (the frame's row of the
// caller's camera table, already in the frame's shared scratch).
template <typename E, int LANES = 32, bool FRAME_CAMERA = false>
__device__ __forceinline__ void okp_group_frame(const int n, const int lane, const OkpGroupScratch& g, const OkpGroupArgs& a,
                                                const OkpDecodeTables& t, const OkpCamera* frame_camera = nullptr) {
    constexpr int THREADS = LANES;
    const OkpCamera& cam = FRAME_CAMERA ? *frame_camera : a.cam;
    const unsigned FULL = LANES == 32 ? 0xffffffffu : (0xffffu << (threadIdx.x & 16));
    const bool CLEAR = a.prm.lean_tables == 0;
    const int C = a.C, H = a.H, W = a.W, S = a.S;
    const int K = a.prm.max_peaks, O = a.prm.max_objects, V = a.prm.max_votes, T = C - 1;
    const size_t HW = (size_t)H * W;
    const size_t m0 = (size_t)n * C;
    const E* depth = reinterpret_cast<const E*>(a.depth);
    const E* centers = reinterpret_cast<const E*>(a.centers);
    unsigned int& s_flags = *g.flags;
    const int* s_counts = g.counts;
    const unsigned lt = ((1u << (threadIdx.x & 31)) - 1u) & FULL;      // the frame's lanes below this one

    const int n_center = s_counts[0];
    const int n_obj = n_center < O ? n_center : O;
    if (CLEAR) {
        // reset this frame's object tables (flat, coalesced; every region is contiguous per frame)
        const int oc = O * C, ocs = oc * S;
        int32_t* assigned = t.kp_assigned + (size_t)n * oc;
        int32_t* count = t.kp_count + (size_t)n * oc;
        for (int i = lane; i < oc; i += THREADS) { assigned[i] = 0; count[i] = 0; }
        int32_t* peak = t.kp_peak + (size_t)n * ocs;
        for (int i = lane; i < ocs; i += THREADS) peak[i] = -1;
        float2* xy = reinterpret_cast<float2*>(t.kp_xy) + (size_t)n * ocs;
        for (int i = lane; i < ocs; i += THREADS) xy[i] = make_float2(0.0f, 0.0f);
        double* point = t.kp_point + (size_t)n * ocs * 3;
        for (int i = lane; i < ocs * 3; i += THREADS) point[i] = 0.0;
        int32_t* nv = t.n_votes + (size_t)n * O;
        for (int i = lane; i < O; i += THREADS) nv[i] = 0;
        double2* votes = reinterpret_cast<double2*>(t.votes) + (size_t)n * O * V;
        for (int i = lane; i < O * V; i += THREADS) votes[i] = make_double2(0.0, 0.0);
    }
    if (n_center == 0) {                                   // pipeline.py:105-106
        if (lane == 0) {
            const unsigned int f = s_flags | OKP_FLAG_NO_CENTERS;
            t.n_objects[n] = 0; t.flags[n] = f;
            okp_record_header(a.sinks, n, 0, f);
        }
        return;
    }
    if (lane == 0) {
        if (n_center > O) atomicOr(&s_flags, OKP_FLAG_OBJECT_OVERFLOW);
        int at = 0;
        for (int c = 0; c < C; ++c) { g.start[c] = at; at += s_counts[c]; }
        g.start[C] = at;
    }
    // ---- centre peaks become objects (pipeline.py:109-114) ----
    for (int k = lane; k < n_center; k += THREADS) {
        const int o = k < n_obj ? k : -1;
        g.obj[k] = o;
        if (o >= 0) { g.center[o][0] = (double)g.xy[2 * k]; g.center[o][1] = (double)g.xy[2 * k + 1]; }
        t.peak_object[m0 * K + k] = o;
    }
    for (int i = lane; i < n_obj * C; i += THREADS) g.assigned[i] = 0;
    for (int o = lane; o < n_obj; o += THREADS) g.nvotes[o] = 0;
    __syncwarp(FULL);
    const int total = g.start[C];

    // ---- pass 1: spoke peaks vote for a centre (pipeline.py:115-128); vote-list slots and (object, map) ranks ----
    for (int base = g.start[1]; base < total; base += THREADS) {
        const int idx = base + lane;
        const bool active = idx < total;
        int c = 1, i = 0, arg = -1;
        double vx = 0.0, vy = 0.0;
        if (active) {
            while (idx >= g.start[c + 1]) ++c;
            const int k = idx - g.start[c];
            i = c * K + k;
            const size_t s = (m0 + c) * K + k;
            const float px = g.xy[2 * i], py = g.xy[2 * i + 1];
            const int xi = okp_clamp(__float2int_rn(px), 0, W - 1);       // np.round = half to even
            const int yi = okp_clamp(__float2int_rn(py), 0, H - 1);
            const E* cmap = centers + ((size_t)n * T + (c - 1)) * 2 * HW;
            vx = ((double)xi + 0.5) + (double)okp_ld<E>(cmap + (size_t)yi * W + xi);
            vy = ((double)yi + 0.5) + (double)okp_ld<E>(cmap + HW + (size_t)yi * W + xi);
            g.vote[2 * i] = vx; g.vote[2 * i + 1] = vy;
            reinterpret_cast<double2*>(t.peak_vote)[s] = make_double2(vx, vy);
            // nearest centre = first minimum of sqrt(d2) like np.argmin over np.linalg.norm. sqrt is monotone, so the
            // minimum is sqrt(min d2); it is attained by every object whose d2 rounds to the same square root, i.e. whose
            // d2 lies within a few ulp of the minimum: only those need their own square root
            double m2 = 0.0;
            for (int o = 0; o < n_obj; ++o) {
                const double dx = g.center[o][0] - vx, dy = g.center[o][1] - vy;
                const double d2 = dx * dx + dy * dy;
                if (o == 0 || d2 < m2) m2 = d2;
            }
            const double dmin = sqrt(m2);
            const double near = m2 * (1.0 + 1e-15);
            for (int o = 0; o < n_obj; ++o) {
                const double dx = g.center[o][0] - vx, dy = g.center[o][1] - vy;
                const double d2 = dx * dx + dy * dy;
                if (d2 == m2 || (d2 <= near && sqrt(d2) == dmin)) { arg = o; break; }
            }
            if (dmin > a.prm.outlier_distance) {
                atomicOr(&s_flags, OKP_FLAG_OUTLIER_SKIPPED);              // the reference prints and skips
                arg = -1;
            }
            g.obj[i] = arg;
            t.peak_object[s] = arg;
        }
        const bool member = active && arg >= 0;
        const unsigned same_o = __match_any_sync(FULL, member ? arg : (int)(0x80000000u | (unsigned)lane));
        const unsigned same_oc = __match_any_sync(FULL, member ? ((c << 8) | arg) : (int)(0x80000000u | (unsigned)lane));
        int r_o = 0, r_oc = 0;
        if (member) {
            r_o = __popc(same_o & lt);
            r_oc = __popc(same_oc & lt);
            const int slot = g.nvotes[arg] + r_o;                          // assignment order: map-major, raster inside a map
            if (slot < V) reinterpret_cast<double2*>(t.votes)[((size_t)n * O + arg) * V + slot] = make_double2(vx, vy);
            else atomicOr(&s_flags, OKP_FLAG_VOTE_OVERFLOW);
            g.rank[i] = g.assigned[arg * C + c] + r_oc;
        }
        __syncwarp(FULL);
        if (member) {
            if (r_o == 0) g.nvotes[arg] += __popc(same_o);
            if (r_oc == 0) g.assigned[arg * C + c] += __popc(same_oc);
        }
        __syncwarp(FULL);
    }
    for (int o = lane; o < n_obj; o += THREADS) t.n_votes[(size_t)n * O + o] = g.nvotes[o];

    // ---- per (object, map): counts; the over-detection cases are resolved (and lifted) here, one lane each ----
    for (int i = lane; i < n_obj * C; i += THREADS) {
        const int o = i / C, c = i - o * C;
        const size_t oc = ((size_t)n * O + o) * C + c;
        const int limit = a.config.cfg[c];
        const int cnt = c == 0 ? 1 : g.assigned[i];
        t.kp_assigned[oc] = cnt;
        if (cnt <= limit) {                                // everything is kept (pass 2); cnt == 0: pipeline.py:150-152
            if (cnt > 0 || !CLEAR) t.kp_count[oc] = cnt;
            okp_record_count(a.sinks, n, O, C, o, c, cnt);
            continue;
        }
        const int* obj = g.obj + c * K;
        const float* xy = g.xy + (size_t)c * K * 2;
        float pts[OKP_MAX_SLOTS][2];
        int ids[OKP_MAX_SLOTS];
        int kept = 0;
        if (limit == 1) {                                  // pipeline.py:139-142: most confident detection
            int arg = -1;
            float best = 0.0f;
            for (int k = 0; k < s_counts[c]; ++k)
                if (obj[k] == o) {
                    const float conf = g.conf[c * K + k];
                    if (arg < 0 || conf > best) { best = conf; arg = k; }   // first maximum, like np.argmax
                }
            ids[0] = arg;
            pts[0][0] = xy[2 * arg];
            pts[0][1] = xy[2 * arg + 1];
            kept = 1;
            atomicOr(&s_flags, OKP_FLAG_ARGMAX_RESOLVED);
        } else {                                           // pipeline.py:143-148: cluster
            unsigned char members[OKP_MAX_PEAKS];
            int m = 0;
            for (int k = 0; k < s_counts[c]; ++k)
                if (obj[k] == o) members[m++] = (unsigned char)k;
            kept = limit;
            okp_cluster_detections(xy, members, m, kept, a.prm.kmeans_iterations, &pts[0][0]);
            for (int s = 0; s < kept; ++s) ids[s] = -1;
            atomicOr(&s_flags, OKP_FLAG_CLUSTERED);
        }
        t.kp_count[oc] = kept;
        okp_record_count(a.sinks, n, O, C, o, c, kept);
        for (int s = 0; s < kept; ++s) {
            t.kp_peak[oc * S + s] = ids[s];
            reinterpret_cast<float2*>(t.kp_xy)[oc * S + s] = make_float2(pts[s][0], pts[s][1]);
            double p3[3] = {0.0, 0.0, 0.0};
            if (a.have_camera) {
                okp_detection_to_point(pts[s][0], pts[s][1], depth + (m0 + c) * HW, H, W, cam, a.prm.compat_clip_bug, p3);
                double* out = t.kp_point + (oc * S + s) * 3;
                out[0] = p3[0]; out[1] = p3[1]; out[2] = p3[2];
            }
            okp_record_point(a.sinks, n, O, C, a.P, a.config, o, c, s, p3);
        }
    }

    // ---- pass 2: every kept peak writes its keypoint slot and lifts itself to 3D (pipeline.py:164-171, 189-199); the
    // point goes to the table and, when the caller asked for them, into the compact record of every sink ----
    for (int base = 0; base < total; base += THREADS) {
        const int idx = base + lane;
        if (idx >= total) continue;
        int c = 0;
        while (idx >= g.start[c + 1]) ++c;
        const int k = idx - g.start[c];
        const int i = c * K + k;
        const int o = g.obj[i];
        if (o < 0) continue;
        int slot = 0;
        if (c > 0) {
            if (g.assigned[o * C + c] > a.config.cfg[c]) continue;     // resolved above
            slot = g.rank[i];
        }
        const size_t ocs = (((size_t)n * O + o) * C + c) * S + slot;
        const float px = g.xy[2 * i], py = g.xy[2 * i + 1];
        t.kp_peak[ocs] = k;
        reinterpret_cast<float2*>(t.kp_xy)[ocs] = make_float2(px, py);
        double p3[3] = {0.0, 0.0, 0.0};
        if (a.have_camera) {
            okp_detection_to_point(px, py, depth + (m0 + c) * HW, H, W, cam, a.prm.compat_clip_bug, p3);
            double* out = t.kp_point + ocs * 3;
            out[0] = p3[0]; out[1] = p3[1]; out[2] = p3[2];
        }
        okp_record_point(a.sinks, n, O, C, a.P, a.config, o, c, slot, p3);
    }
    __syncwarp(FULL);
    if (lane == 0) {
        const unsigned int f = s_flags;
        t.n_objects[n] = n_obj; t.flags[n] = f;
        okp_record_header(a.sinks, n, n_obj, f);
    }
}

// Stand-alone form: one warp per frame, four frames per CTA (an SM holds 64 frames whose latency chains overlap).
// The frame's peak records are pulled from the tables into shared memory with one round trip. only_pending != 0: only
// frames marked OKP_GROUP_PENDING by the fused decode kernel are processed (the fix-up launch: with no overflowing map
// it is one read of n_objects per frame). okp_group_cameras_kernel below repeats these first steps (flags, counts, the
// pull of the peak records): a change to one of the two belongs in the other.
template <typename E, int LANES>
__global__ void __launch_bounds__(128)
okp_group_kernel(const __grid_constant__ OkpGroupArgs a, const int only_pending, const OkpDecodeTables t) {
    constexpr int SHIFT = LANES == 32 ? 5 : 4;
    const int lane = threadIdx.x & (LANES - 1);
    const unsigned mask = LANES == 32 ? 0xffffffffu : (0xffffu << (threadIdx.x & 16));
    const int n = blockIdx.x * (blockDim.x >> SHIFT) + (threadIdx.x >> SHIFT);
    okp_wait_for_predecessor();                           // launched as a programmatic dependent of the peak / fix-up kernel
    if (n >= a.N) return;
    if (only_pending && t.n_objects[n] != OKP_GROUP_PENDING) return;
    const int C = a.C, K = a.prm.max_peaks, O = a.prm.max_objects;
    extern __shared__ __align__(16) unsigned char group_smem[];
    const OkpGroupScratch g = okp_group_scratch(group_smem + (size_t)(threadIdx.x >> SHIFT) * a.frame_smem_bytes, C, K, O);
    const size_t m0 = (size_t)n * C;
    // OKP_FLAG_GENERIC_PATH is a property of the call, written by the peak extraction: keep it
    if (lane == 0) *g.flags = t.flags[n] & OKP_FLAG_GENERIC_PATH;
    __syncwarp(mask);
    if (lane < C) {
        const int c = t.peak_count[m0 + lane];
        g.counts[lane] = c < K ? c : K;
        if (c > K) atomicOr(g.flags, OKP_FLAG_PEAK_OVERFLOW);
    }
    __syncwarp(mask);
    for (int i = lane; i < C * K; i += LANES) {
        const int c = i / K, k = i - c * K;
        if (k >= g.counts[c]) continue;
        const size_t s = (m0 + c) * K + k;
        const float2 p = *reinterpret_cast<const float2*>(t.peak_xy + 2 * s);
        g.xy[2 * i] = p.x; g.xy[2 * i + 1] = p.y;
        g.conf[i] = t.peak_conf[s];
    }
    __syncwarp(mask);
    okp_group_frame<E, LANES>(n, lane, g, a, t);
}

// Per-frame cameras (okp_decode_cameras_*, okp_group_objects_cameras_*): okp_group_kernel's steps, except that the frame's
// lanes first copy cameras[n] (device memory, 16-byte aligned: 9 words of 16 bytes) into the last bytes of the frame's
// scratch (okp_group_smem_bytes(..., true)) and the 3D lift reads that copy instead of a.cam, which is not read. Never a
// fix-up launch: the fused single pass has no per-frame-camera form. A kernel of its own rather than a template flag of
// okp_group_kernel: any rewrapping of that kernel's body changes its register allocation and scheduling.
// Registers: under __launch_bounds__(128) alone ptxas settles on 64 (32 lanes) / 72 (16 lanes) and reloads loop invariants
// from the stack in every iteration of pass 2, the per-peak lift loop. 72 registers keep pass 2 free of spills in both
// forms (the remaining few spill bytes sit around the clustering call); a 128-thread CTA still fits 7 times per SM by
// registers, and the 16-lane form (8 frames per CTA) is limited by shared memory first.
template <typename E, int LANES>
__global__ void __maxnreg__(72)
okp_group_cameras_kernel(const __grid_constant__ OkpGroupArgs a, const OkpDecodeTables t, const OkpCamera* __restrict__ cameras) {
    constexpr int SHIFT = LANES == 32 ? 5 : 4;
    constexpr int WORDS = (int)(sizeof(OkpCamera) / sizeof(uint4));
    const int lane = threadIdx.x & (LANES - 1);
    const unsigned mask = LANES == 32 ? 0xffffffffu : (0xffffu << (threadIdx.x & 16));
    const int n = blockIdx.x * (blockDim.x >> SHIFT) + (threadIdx.x >> SHIFT);
    okp_wait_for_predecessor();
    if (n >= a.N) return;
    const int C = a.C, K = a.prm.max_peaks, O = a.prm.max_objects;
    extern __shared__ __align__(16) unsigned char group_smem[];
    unsigned char* const mine = group_smem + (size_t)(threadIdx.x >> SHIFT) * a.frame_smem_bytes;
    const OkpGroupScratch g = okp_group_scratch(mine, C, K, O);
    OkpCamera* const camera = reinterpret_cast<OkpCamera*>(mine + a.frame_smem_bytes - sizeof(OkpCamera));
    if (lane < WORDS) reinterpret_cast<uint4*>(camera)[lane] = __ldg(reinterpret_cast<const uint4*>(cameras + n) + lane);
    const size_t m0 = (size_t)n * C;
    if (lane == 0) *g.flags = t.flags[n] & OKP_FLAG_GENERIC_PATH;
    __syncwarp(mask);
    if (lane < C) {
        const int c = t.peak_count[m0 + lane];
        g.counts[lane] = c < K ? c : K;
        if (c > K) atomicOr(g.flags, OKP_FLAG_PEAK_OVERFLOW);
    }
    __syncwarp(mask);
    for (int i = lane; i < C * K; i += LANES) {
        const int c = i / K, k = i - c * K;
        if (k >= g.counts[c]) continue;
        const size_t s = (m0 + c) * K + k;
        const float2 p = *reinterpret_cast<const float2*>(t.peak_xy + 2 * s);
        g.xy[2 * i] = p.x; g.xy[2 * i + 1] = p.y;
        g.conf[i] = t.peak_conf[s];
    }
    __syncwarp(mask);
    okp_group_frame<E, LANES, true>(n, lane, g, a, t, camera);
}
