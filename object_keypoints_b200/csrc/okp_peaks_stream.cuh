// okp_peaks_stream.cuh -- persistent, warp-specialised form of the strip kernel (okp_peaks_strip.cuh).
//
// Same arithmetic (okp_strip_step / okp_strip_batch, the bounded filter + exact check) and the same
// shared-memory stage layout, different control flow. The one-shot kernel gives every group of M maps its
// own CTA: mbarrier set-up, a pipeline fill, the streaming phase, and then an epilogue (exact box sums of
// the candidates, ordering, table writes) during which the CTA's TMA pipeline is empty and its compute
// warps are idle at four __syncthreads. At 180x320 that is ~8 % of a CTA's life, at the network's 64x64
// (14 row batches per map) it is half of it (profiles/r01f_k1_ncu.md: 0.38 of the HBM peak).
//
// Here a CTA is resident for the whole launch and walks over groups g = blockIdx.x, + gridDim.x, ...:
//   * the producer lane streams the batches of consecutive groups back to back (the ring of NS stages
//     never drains between groups);
//   * the compute warps go from the last batch of a group straight into the first batch of the next; their
//     candidates go into one of two candidate buffers;
//   * epilogue warps consume a finished buffer (exact sums from L2, undecided neighbours, raster ranks,
//     table writes) WHILE the compute warps stream the next group. Hand-over is one mbarrier arrive per
//     warp per group (cand_full / cand_free), not per row batch, so it costs nothing (the r01b design paid
//     42 % of its issue slots for per-batch hand-over spins).
//
// FUSED = true (round 2; okp_decode_*): a group is a whole number of frames (M = F * C maps) and the epilogue warps go
// on from the frame's sorted peak list -- still in shared memory -- to the grouping and the 3D lift (okp_group_frame,
// okp_group.cuh) and to the frame's compact record (okp_records.cuh), so that ObjectKeypointPipeline.__call__
// (perception/pipeline.py:182-200) is ONE streaming pass over the heatmaps: no second kernel that re-reads the peak
// tables, no pack kernel for the multi-GPU gather. A frame one of whose maps overflowed (more than K peaks, negative /
// NaN values, more candidates than slots) is marked OKP_GROUP_PENDING and finished by the fix-up launches
// (okp_peaks_overflow_kernel, okp_group_kernel with only_pending).
#pragma once
#include "okp_peaks_strip.cuh"
#include "okp_group.cuh"

struct OkpStreamPlan {
    OkpStripPlan s;               // geometry, M, NS, stage layout
    int groups;                   // ceil(maps / M)
    int EW;                       // epilogue warps
    int off_pending[2], off_count[2];   // candidate lists and [n_pending[M], redo[M]] per buffer
    int off_peaks, off_items, off_misc, off_mbar;
    int off_group;                // fused: F frame scratches of okp_group_smem_bytes() (okp_group.cuh)
    int C;                        // maps per frame
    int F;                        // fused: frames per group (M = F * C); 0 = peaks only
    int lean;                     // OkpDecodeParams.lean_tables
    int smem_bytes;
    int threads;                  // compute warps + producer warp + epilogue warps
};

__device__ __forceinline__ void okp_named_barrier(int id, int threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// The epilogue warps' loop of the stream kernel below: one finished candidate buffer at a time -- exact box sums from L2,
// undecided neighbours, raster ranks, table rows and, fused, the frame's grouping and 3D lift. et: thread index among the
// sp.EW epilogue warps. The CTA's groups are the ones its producer lane claimed from the launch's counter (ids in the ring
// behind the mbarriers, -1 = no more).
template <typename T, bool FUSED>
__device__ __forceinline__ void okp_stream_epilogue(unsigned char* smem, const OkpStreamPlan& sp, const T* __restrict__ heat,
                                                    const float threshold, const OkpDecodeTables& t, const OkpGroupArgs& ga,
                                                    const int et) {
    const OkpStripPlan& p = sp.s;
    const int H = p.H, W = p.W;
    OkpStripPeak* peaks = reinterpret_cast<OkpStripPeak*>(smem + sp.off_peaks);                // [M][PK]
    uint32_t* items = reinterpret_cast<uint32_t*>(smem + sp.off_items);                        // [IC]
    int* n_peaks = reinterpret_cast<int*>(smem + sp.off_misc);                                 // [M]
    int* n_items = n_peaks + p.M;                                                              // [1]
    int* cand_start = n_items + 1;                                                             // [M + 1] prefix of candidate counts
    int* pend = cand_start + p.M + 1;                                                          // [M] fused: frame f is left to the fix-up launches
    uint64_t* cand_full = reinterpret_cast<uint64_t*>(smem + sp.off_mbar) + 2 * OKP_STRIP_MAX_NS;
    uint64_t* cand_free = cand_full + 2;
    const volatile int* group_ring = reinterpret_cast<const volatile int*>(cand_free + 2);    // [8] claimed group ids
    const int ethreads = sp.EW * 32;
    for (int it = 0;; ++it) {
        const int buf = it & 1;
        okp_mbar_wait(cand_full + buf, (uint32_t)((it >> 1) & 1), 400);
        const int group = group_ring[it & 7];
        if (group < 0) break;                                                                  // the end marker
        const int first_map = group * p.M;
        OkpStripCandidate* pending = reinterpret_cast<OkpStripCandidate*>(smem + sp.off_pending[buf]);
        int* n_pending = reinterpret_cast<int*>(smem + sp.off_count[buf]);
        int* redo = n_pending + p.M;

        // candidates are few and sit at the front of each map's list: index them densely so that every
        // lane has one (all loads of a pass in flight together) instead of walking M * PK mostly empty slots
        if (et == 0) {
            int at = 0;
            for (int mm = 0; mm < p.M; ++mm) {
                cand_start[mm] = at;
                at += first_map + mm < p.maps ? okp_min(n_pending[mm], p.PK) : 0;
            }
            cand_start[p.M] = at;
        }
        okp_named_barrier(1, ethreads);
        const int candidates = cand_start[p.M];

        // A: exact box sum (the reference's raster-order adds) and centroid of every candidate
        for (int idx = et; idx < candidates; idx += ethreads) {
            int lo = 0, hi = p.M;                                 // last mm with cand_start[mm] <= idx
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (cand_start[mid] <= idx) lo = mid; else hi = mid; }
            const int mm = lo, i = mm * p.PK + (idx - cand_start[mm]);
            OkpStripPeak pk;
            pk.key = -1; pk.score = 0.0f; pk.cx = 0.0f; pk.cy = 0.0f; pk.conf = 0.0f;
            {
                const OkpStripCandidate cd = pending[i];
                const int y = cd.key / W, x = cd.key - y * W;
                const T* src = heat + (size_t)(first_map + mm) * H * W;
                float q[25];
                // almost every candidate is an interior pixel: 25 unconditional loads at constant offsets
                // (a fifth of the instructions of the border-checked form, which matters because the
                // epilogue warps are latency-bound: profiles/r01m_k1_64x64_ncu.md)
                const bool interior = y >= 2 && y + 2 < H && x >= 2 && x + 2 < W;
                if (interior) {
                    const T* corner = src + (size_t)(y - 2) * W + (x - 2);
#pragma unroll
                    for (int k = 0; k < 25; ++k) q[k] = okp_ld<T>(corner + (size_t)(k / 5) * W + k % 5);
                } else {
#pragma unroll
                    for (int k = 0; k < 25; ++k) {
                        const int i2 = y + k / 5 - 2, j2 = x + k % 5 - 2;
                        const bool in = i2 >= 0 && i2 < H && j2 >= 0 && j2 < W;
                        q[k] = in ? okp_ld<T>(src + (size_t)i2 * W + j2) : 0.0f;
                    }
                }
                float sum = 0.0f;
#pragma unroll
                for (int k = 0; k < 25; ++k) sum = __fadd_rn(sum, q[k]);
                if (sum > threshold) {
                    float sy = 0.0f, sx = 0.0f, spr = 0.0f;
                    if (interior) {                           // same operations in the same order, nothing masked
#pragma unroll
                        for (int k = 0; k < 25; ++k) {
                            sy = __fadd_rn(sy, __fmul_rn(q[k], (float)(y + k / 5 - 2)));
                            sx = __fadd_rn(sx, __fmul_rn(q[k], (float)(x + k % 5 - 2)));
                            spr = __fadd_rn(spr, q[k]);
                        }
                    } else {
#pragma unroll
                        for (int k = 0; k < 25; ++k) {
                            const int i2 = y + k / 5 - 2, j2 = x + k % 5 - 2;
                            const bool in = i2 >= 0 && i2 < H && j2 >= 0 && j2 < W;
                            if (in) {
                                sy = __fadd_rn(sy, __fmul_rn(q[k], (float)i2));
                                sx = __fadd_rn(sx, __fmul_rn(q[k], (float)j2));
                                spr = __fadd_rn(spr, q[k]);
                            }
                        }
                    }
                    pk.key = cd.key;
                    pk.score = sum;
                    pk.cx = __fdiv_rn(sx, spr);
                    pk.cy = __fdiv_rn(sy, spr);
                    pk.conf = spr;
                    uint32_t ties = cd.ties;
                    ties &= (y >= 2 ? 0x1Fu : 0u) | (y >= 1 ? 0x3E0u : 0u) | 0x6C00u | (y + 1 < H ? 0xF8000u : 0u) | (y + 2 < H ? 0x1F00000u : 0u);
                    ties &= (x >= 2 ? 0x108421u : 0u) | (x >= 1 ? 0x210842u : 0u) | 0x421084u | (x + 1 < W ? 0x842108u : 0u) | (x + 2 < W ? 0x1084210u : 0u);
                    if (ties) {
                        const int at = atomicAdd(n_items, __popc(ties));
                        if (at + __popc(ties) > p.IC) {
                            redo[mm] = 1;
                            for (int n = at; n < p.IC; ++n) items[n] = 0xFFFFFFFFu;
                        } else {
                            int n = at;
                            while (ties) {
                                const int k = __ffs(ties) - 1;
                                ties &= ties - 1;
                                items[n++] = ((uint32_t)i << 5) | (uint32_t)k;
                            }
                        }
                    }
                }
            }
            peaks[i] = pk;
        }
        okp_named_barrier(1, ethreads);

        // B: undecided neighbours -- exact box sum against the candidate's
        {
            const int total_items = okp_min(*n_items, p.IC);
            for (int n = et; n < total_items; n += ethreads) {
                const uint32_t item = items[n];
                if (item == 0xFFFFFFFFu) continue;
                const int i = (int)(item >> 5), k = (int)(item & 31u);
                const int mm = i / p.PK;
                const int key = pending[i].key;
                const int y = key / W, x = key - y * W;
                const T* src = heat + (size_t)(first_map + mm) * H * W;
                if (okp_exact_box_sum<T>(src, H, W, y + k / 5 - 2, x + k % 5 - 2) > peaks[i].score) peaks[i].key = -1;
            }
        }
        okp_named_barrier(1, ethreads);
        for (int idx = et; idx < candidates; idx += ethreads) {
            int lo = 0, hi = p.M;
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (cand_start[mid] <= idx) lo = mid; else hi = mid; }
            if (peaks[lo * p.PK + (idx - cand_start[lo])].key >= 0) atomicAdd(n_peaks + lo, 1);
        }
        okp_named_barrier(1, ethreads);

        // C: raster order (rank by key), final tables, unused slots cleared (not with lean tables). Fused: the sorted
        // rows also go into the frame's grouping scratch, which is what phase D works from.
        const int K = p.K;
        for (int mm = 0; mm < p.M && first_map + mm < p.maps; ++mm) {
            const int map = first_map + mm;
            const int total = (redo[mm] || n_pending[mm] > p.PK) ? K + 1 : n_peaks[mm];
            if (et == 0) {
                t.peak_count[map] = total;
                if (FUSED) {
                    const int f = mm / sp.C, c = mm - f * sp.C;
                    const OkpGroupScratch g = okp_group_scratch(smem + sp.off_group + (size_t)f * ga.frame_smem_bytes, sp.C, K,
                                                                ga.prm.max_objects);
                    g.counts[c] = total < K ? total : K;
                    if (c == 0) *g.flags = 0;
                    if (total > K) pend[f] = 1;
                } else if (t.flags && map % sp.C == 0) {
                    t.flags[map / sp.C] = 0;                 // a stale OKP_FLAG_GENERIC_PATH must not survive (okp_group_kernel keeps the bit)
                }
            }
            if (total > K || sp.lean) continue;              // tables of an overflowing map are written by the overflow path
            for (int slot = et; slot < K; slot += ethreads) {
                const size_t dst = (size_t)map * K + slot;
                t.peak_object[dst] = -1;
                reinterpret_cast<double2*>(t.peak_vote)[dst] = make_double2(0.0, 0.0);
                if (slot >= total) {
                    reinterpret_cast<int2*>(t.peak_yx)[dst] = make_int2(-1, -1);
                    t.peak_score[dst] = 0.0f;
                    reinterpret_cast<float2*>(t.peak_xy)[dst] = make_float2(0.0f, 0.0f);
                    t.peak_conf[dst] = 0.0f;
                }
            }
        }
        for (int idx = et; idx < candidates; idx += ethreads) {
            int lo = 0, hi = p.M;
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (cand_start[mid] <= idx) lo = mid; else hi = mid; }
            const int mm = lo, i = mm * p.PK + (idx - cand_start[mm]);
            const OkpStripPeak pk = peaks[i];
            if (pk.key < 0) continue;
            if (redo[mm] || n_pending[mm] > p.PK || n_peaks[mm] > K) continue;
            const OkpStripPeak* mine = peaks + (size_t)mm * p.PK;
            const int np = n_pending[mm];
            int rank = 0;
            for (int j = 0; j < np; ++j) { const int kj = mine[j].key; rank += (kj >= 0 && kj < pk.key); }
            const size_t dst = (size_t)(first_map + mm) * K + rank;
            const int y = pk.key / W;
            reinterpret_cast<int2*>(t.peak_yx)[dst] = make_int2(y, pk.key - y * W);
            t.peak_score[dst] = pk.score;
            reinterpret_cast<float2*>(t.peak_xy)[dst] = make_float2(pk.cx, pk.cy);
            t.peak_conf[dst] = pk.conf;
            if (sp.lean) {                                   // the row's assignment columns, which the clearing loop did not reset
                t.peak_object[dst] = -1;
                reinterpret_cast<double2*>(t.peak_vote)[dst] = make_double2(0.0, 0.0);
            }
            if (FUSED) {
                const int f = mm / sp.C, c = mm - f * sp.C;
                const OkpGroupScratch g = okp_group_scratch(smem + sp.off_group + (size_t)f * ga.frame_smem_bytes, sp.C, K,
                                                            ga.prm.max_objects);
                g.xy[2 * (c * K + rank)] = pk.cx; g.xy[2 * (c * K + rank) + 1] = pk.cy;
                g.conf[c * K + rank] = pk.conf;
            }
        }
        okp_named_barrier(1, ethreads);
        // hand the candidate buffer back, cleared: the compute warps never wait for the grouping below
        for (int i = et; i < 2 * p.M; i += ethreads) n_pending[i] = 0;
        for (int i = et; i < p.M + 1; i += ethreads) n_peaks[i] = 0;
        okp_named_barrier(1, ethreads);
        if ((et & 31) == 0) okp_mbar_arrive(cand_free + buf);

        // D (fused): grouping + 3D lift + compact record, one warp per frame, from the sorted peak list in shared memory
        if (FUSED) {
            const int first_frame = first_map / sp.C;
            for (int f = et >> 5; f < sp.F && first_frame + f < ga.N; f += sp.EW) {
                const int n = first_frame + f;
                if (pend[f]) {                               // okp_group_kernel keeps OKP_FLAG_GENERIC_PATH: not from this call
                    if ((et & 31) == 0) { t.n_objects[n] = OKP_GROUP_PENDING; t.flags[n] = 0; }
                } else {
                    const OkpGroupScratch g = okp_group_scratch(smem + sp.off_group + (size_t)f * ga.frame_smem_bytes, sp.C, K,
                                                                ga.prm.max_objects);
                    okp_group_frame<T>(n, et & 31, g, ga, t);
                }
            }
            okp_named_barrier(1, ethreads);                  // phase C of the next group rewrites the scratches
            for (int i = et; i < p.M; i += ethreads) pend[i] = 0;
        }
    }
}

template <typename T, bool FUSED>
// 96 registers: two CTAs of 320 threads per SM (__maxnreg__ and __launch_bounds__ exclude each other; the launch uses at
// most OKP_STRIP_MAX_THREADS = 640 threads, which 96 registers also allow)
__global__ void __maxnreg__(96)
okp_peaks_stream_kernel(const __grid_constant__ CUtensorMap tmap, const T* __restrict__ heat, const __grid_constant__ OkpStreamPlan sp,
                        float threshold, float thr_lo, const __grid_constant__ OkpDecodeTables t,
                        const __grid_constant__ OkpGroupArgs ga, int* __restrict__ group_counter) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int RB = OKP_STRIP_RB;
    const OkpStripPlan& p = sp.s;
    const int NS = p.NS;
    int* n_peaks = reinterpret_cast<int*>(smem + sp.off_misc);              // [M] + n_items [1] + cand_start [M + 1] + pend [M]: the
    int* pend = n_peaks + 2 * p.M + 2;                                      // epilogue's (okp_stream_epilogue), zeroed here
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + sp.off_mbar);       // [NS] TMA landed
    uint64_t* done = full + OKP_STRIP_MAX_NS;                               // [NS] compute warps finished the batch
    uint64_t* cand_full = done + OKP_STRIP_MAX_NS;                          // [2] candidate buffer complete
    uint64_t* cand_free = cand_full + 2;                                    // [2] epilogue finished with the buffer
    volatile int* group_ring = reinterpret_cast<volatile int*>(cand_free + 2);   // [8] group id of iteration it (it & 7), -1 = end

    const int tid = threadIdx.x;
    const int H = p.H, W = p.W;
    const int compute_warps = (p.threads + 31) >> 5;
    const int warp = tid >> 5;

    for (int b = 0; b < 2; ++b) {
        int* count = reinterpret_cast<int*>(smem + sp.off_count[b]);
        for (int i = tid; i < 2 * p.M; i += blockDim.x) count[i] = 0;
    }
    for (int i = tid; i < p.M + 1; i += blockDim.x) n_peaks[i] = 0;
    for (int i = tid; i < p.M; i += blockDim.x) pend[i] = 0;
    if (tid == 0) {
        for (int i = 0; i < NS; ++i) { okp_mbar_init(full + i, 1); okp_mbar_init(done + i, compute_warps); }
        for (int i = 0; i < 2; ++i) { okp_mbar_init(cand_full + i, compute_warps); okp_mbar_init(cand_free + i, sp.EW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    // Groups are CLAIMED from a counter of the launch (zeroed by the caller), one at a time, by the producer lane: a CTA
    // that becomes resident late -- another kernel held its SM, e.g. the exchange barrier of the previous step beside a
    // multi-GPU decode -- simply takes fewer groups. With the static round-robin of round 1 such a CTA delayed the whole
    // launch by its lag (K1 stretched 479 -> 518 us on 8 GPUs). The id travels to the compute warps behind the `full`
    // barrier of the group's first batch and to the epilogue warps behind `cand_full`; -1 ends the roles' loops.
    if (warp == compute_warps) {
        // ------------------------------- producer: one lane, batches of consecutive groups back to back ---
        if ((tid & 31) == 0) {
            const CUtensorMap* tmap_ptr = &tmap;
            int stage = 0;
            uint32_t parity = 0;
            long long q = 0;
            for (int it = 0;; ++it) {
                int group = atomicAdd(group_counter, 1);
                if (group >= sp.groups) group = -1;
                group_ring[it & 7] = group;                   // ordered before the arrive below (release)
                if (group < 0) {                              // end marker: complete the phase the compute warps wait for
                    if (q >= NS) {
                        while (!okp_mbar_try_wait_suspend(done + stage, parity)) {}
                    }
                    okp_mbar_arrive(full + stage);
                    break;
                }
                const int first_map = group * p.M;
                for (int b = 0; b < p.nb; ++b, ++q) {
                    if (q >= NS) {                            // every compute warp has left the stage (sleeps in hardware)
                        while (!okp_mbar_try_wait_suspend(done + stage, parity)) {}
                    }
                    uint64_t* bar = full + stage;
                    unsigned char* dst = smem + (size_t)stage * p.stage_bytes;
                    okp_mbar_expect_tx(bar, (uint32_t)(p.halves * p.half_bytes));
                    okp_tma_load_3d(dst, tmap_ptr, -4 - p.lead[0], b * RB - 2, first_map, bar);
                    if (p.halves == 2)
                        okp_tma_load_3d(dst + p.half_stride, tmap_ptr, 4 * p.half_strips - 4 - p.lead[1], b * RB - 2, first_map, bar);
                    if (++stage == NS) { stage = 0; if (q >= NS) parity ^= 1u; }
                }
            }
        }
    } else if (warp < compute_warps) {
        // ------------------------------- compute warps: the stream ---------------------------------------
        const bool active = tid < p.threads;
        const int ct = active ? tid : p.threads - 1;
        const int mm = ct / p.strips;
        const int s = ct - mm * p.strips;
        const int half = s >= p.half_strips ? 1 : 0;
        OkpStripLane L;
        L.H = H; L.W = W; L.thr_lo = thr_lo; L.PK = p.PK;
        L.xs = 4 * s;
        L.vmask = 0;
#pragma unroll
        for (int c = 0; c < 4; ++c) L.vmask |= (L.xs + c - 2 >= 0 && L.xs + c - 2 < W) ? (1u << c) : 0u;
        if (!active) L.vmask = 0;
        if (active && (tid & 31) > 0 && s > 0) L.vmask |= 16u;
        if (active && (tid & 31) < 31 && s + 1 < p.strips && tid + 1 < p.threads) L.vmask |= 32u;
        const int thread_raw = half * p.half_stride +
                               (mm * RB * p.BW + p.lead[half] + 4 * (s - half * p.half_strips)) * (int)sizeof(T);
        const int row_pitch = p.BW * (int)sizeof(T);
        int stage = 0;
        uint32_t full_parity = 0;
        for (int it = 0;; ++it) {
            const int buf = it & 1;
            if (it >= 2) okp_mbar_wait(cand_free + buf, (uint32_t)(((it >> 1) - 1) & 1));   // the epilogue released the buffer
            okp_mbar_wait(full + stage, full_parity);                 // the group's first batch -- or the end marker
            if (group_ring[it & 7] < 0) {
                __syncwarp();
                if ((tid & 31) == 0) okp_mbar_arrive(cand_full + buf);                      // pass the marker on to the epilogue warps
                break;
            }
            int* count = reinterpret_cast<int*>(smem + sp.off_count[buf]);
            L.pending = reinterpret_cast<OkpStripCandidate*>(smem + sp.off_pending[buf]) + (size_t)mm * p.PK;
            L.n_pending = count + mm;
            float pr[5][4], hp[4], sv[5][4];
            uint32_t sign = 0;
#pragma unroll
            for (int i = 0; i < 5; ++i) {
#pragma unroll
                for (int j = 0; j < 4; ++j) { pr[i][j] = 0.0f; sv[i][j] = -INFINITY; }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) hp[j] = 0.0f;
            for (int b = 0; b < p.nb; ++b) {
                if (b > 0) okp_mbar_wait(full + stage, full_parity);
                const unsigned char* raw = smem + (size_t)stage * p.stage_bytes + thread_raw;
                const int y0 = b * RB - 4;
                if (b >= 2 && y0 + 4 < H)
                    okp_strip_batch<false, T>(raw, row_pitch, pr, hp, sv, sign, y0, L);
                else
                    okp_strip_batch<true, T>(raw, row_pitch, pr, hp, sv, sign, y0, L);
                __syncwarp();
                if ((tid & 31) == 0) okp_mbar_arrive(done + stage);
                if (++stage == NS) { stage = 0; full_parity ^= 1u; }
            }
            if (active && (sign >> 30)) count[p.M + mm] = 1;          // redo (negative, NaN, Inf, >= 2.0): benign race, every writer stores 1
            __syncwarp();
            if ((tid & 31) == 0) okp_mbar_arrive(cand_full + buf);
        }
    } else {
        // ------------------------------- epilogue warps: one finished candidate buffer at a time ---------
        okp_stream_epilogue<T, FUSED>(smem, sp, heat, threshold, t, ga, tid - (compute_warps + 1) * 32);
    }
}

// The stream kernel's plan for `maps` maps of H x W elements of esize bytes (4: float32, 2: bfloat16), K table rows per map,
// C maps per frame; false when the kernel does not cover the shape (the caller runs the generic kernels). group_frame_bytes
// > 0 asks for the fused form: groups of whole frames plus one grouping scratch (group_frame_bytes each) per frame of a
// group; false when not even one frame fits a group (the caller then runs the peak kernel and okp_group_kernel separately).
static inline bool okp_stream_plan(int maps, int C, int H, int W, int K, int esize, int group_frame_bytes, int lean,
                                   OkpStreamPlan* out) {
    const int align = 16 / esize;                         // elements per 16 bytes: TMA box starts and row pitches
    if (maps < 1 || H < 1 || W < 4 || (W % 4) != 0 || (W % align) != 0 || W > 500) return false;
    OkpStreamPlan sp;
    memset(&sp, 0, sizeof(sp));
    OkpStripPlan& p = sp.s;
    p.H = H; p.W = W; p.maps = maps; p.K = K; p.esize = esize;
    p.strips = W / 4 + 1;
    p.lead[0] = align - 4;                                // box 0 starts at column -4 - lead[0] = -align
    if (4 * p.strips + 4 + p.lead[0] <= 256) {
        p.halves = 1; p.half_strips = p.strips;
    } else {
        p.halves = 2; p.half_strips = (p.strips + 1) / 2;
        p.lead[1] = (4 * p.half_strips - 4) % align;      // box 1 starts at the aligned column below 4 * half_strips - 4
    }
    // columns 4s-4 .. 4s+3 of the box's strips behind the lead, rounded up to whole 16-byte units
    p.BW = okp_round_up_int(4 * p.half_strips + 4 + (p.lead[0] > p.lead[1] ? p.lead[0] : p.lead[1]), align);
    if (p.BW > 256) return false;                         // a TMA box holds at most 256 elements per dimension
    p.nb = (H + 6 + OKP_STRIP_RB - 1) / OKP_STRIP_RB;
    p.PK = 2 * K;
    // maps per group, first estimate: as many as the shared-memory budget (110 KB: two CTAs per SM) and 256 compute threads
    // allow, counted with four stages (small maps too) and one candidate buffer; the layout loop below settles it. 256
    // compute threads + the producer warp + one epilogue warp = 320 threads: two CTAs per SM at 96 registers. (288 let a
    // 64x64 bfloat16 plan -- more maps fit its shared-memory budget -- grow to 352 threads, i.e. ONE CTA per SM: 719 us
    // against the float32 plan's 454 us for the same pixels, profiles/r02f_bench_k1.txt)
    const int budget = 110 * 1024;
    const int per_map = 4 * OKP_STRIP_RB * p.BW * p.halves * esize +
                        p.PK * (int)(sizeof(OkpStripCandidate) + sizeof(OkpStripPeak)) + 64 * 4 + 12;
    int M = (budget - 1024) / per_map;
    if (M > 256 / p.strips) M = 256 / p.strips;
    if (M > maps) M = maps;
    if (M < 1) {
        M = 1;
        if (per_map + 1024 > 224 * 1024 || p.strips > OKP_STRIP_MAX_THREADS - 32) return false;
    }
    // small maps (64x64: 14 row batches per group): 224 compute threads leave room for a second epilogue warp inside 320
    // threads, and three stages stream as well as four (r02h / r02i sweeps: 464 -> 440 us float32, 566 -> 505 us bfloat16)
    const bool small_map = p.nb <= 20;
    p.NS = small_map ? 3 : 4;
    if (small_map && M * p.strips > 224) M = 224 / p.strips;
    sp.C = C;
    sp.lean = lean;
    const bool fused = group_frame_bytes > 0;
    if (fused && M < C) return false;
    auto resize = [&](int m) {
        p.M = m;
        p.threads = p.M * p.strips;
        p.IC = p.M * 64;
        p.half_bytes = p.M * OKP_STRIP_RB * p.BW * esize;
        p.half_stride = okp_round_up_int(p.half_bytes, 128);
        p.stage_bytes = p.halves * p.half_stride;
    };
    resize(fused ? M / C * C : M);
    // the second candidate buffer costs PK * 8 bytes per map: give it back from the per-CTA budget by re-planning M
    const int compute_limit = OKP_STRIP_MAX_THREADS - 32 - 2 * 32;   // beside the producer warp and up to two epilogue warps
    for (;;) {
        int off = p.NS * p.stage_bytes;
        for (int b = 0; b < 2; ++b) { sp.off_pending[b] = off; off += p.M * p.PK * (int)sizeof(OkpStripCandidate); }
        sp.off_peaks = off; off += p.M * p.PK * (int)sizeof(OkpStripPeak);
        sp.off_items = off; off += p.IC * 4;
        for (int b = 0; b < 2; ++b) { sp.off_count[b] = off; off += 2 * p.M * 4; }
        sp.off_misc = off; off += (3 * p.M + 2) * 4;
        off = okp_round_up_int(off, 16);
        sp.off_group = off;
        if (fused) off += (p.M / C) * group_frame_bytes;
        sp.off_mbar = off; off += (2 * OKP_STRIP_MAX_NS + 4) * 8 + 32;       // mbarriers + the ring of claimed group ids
        sp.smem_bytes = off;
        const int step = fused ? C : 1;
        if ((off <= budget && p.threads <= compute_limit) || p.M == step) break;
        resize(p.M - step);                                // shrink the group until it fits
    }
    sp.F = fused ? p.M / C : 0;
    if (sp.smem_bytes > 224 * 1024 || p.threads > compute_limit) return false;
    // two epilogue warps where they fit beside the compute warps in 320 threads (two CTAs per SM at 96 registers), else
    // one: small maps (64x64: 14 row batches per group) finish a group every few microseconds and one warp cannot keep
    // up (profiles/r01m_k1_64x64_ncu.md)
    sp.EW = (p.threads + 31) / 32 * 32 + 32 + 64 <= 320 ? 2 : 1;
    sp.groups = (maps + p.M - 1) / p.M;
    sp.threads = (p.threads + 31) / 32 * 32 + 32 + sp.EW * 32;
    *out = sp;
    return true;
}

// ga: grouping arguments (fused form, sp.F > 0) or NULL (peaks only).
template <typename T>
static inline int okp_stream_launch(const T* heat, const OkpStreamPlan& sp, float threshold,
                                    const OkpDecodeTables& tables, const OkpGroupArgs* ga, int* group_counter_dev,
                                    cudaStream_t stream, cudaEvent_t before = nullptr, cudaEvent_t after = nullptr) {
    const OkpStripPlan& p = sp.s;
    OkpEncodeTiledFn encode = okp_encode_tiled_fn();
    if (!encode) return OKP_E_CUDA;
    if (((uintptr_t)heat & 15u) != 0) return OKP_E_UNSUPPORTED;
    CUtensorMap tmap;
    const cuuint64_t dims[3] = {(cuuint64_t)p.W, (cuuint64_t)p.H, (cuuint64_t)p.maps};
    const cuuint64_t strides[2] = {(cuuint64_t)p.W * sizeof(T), (cuuint64_t)p.W * p.H * sizeof(T)};
    const cuuint32_t box[3] = {(cuuint32_t)p.BW, (cuuint32_t)OKP_STRIP_RB, (cuuint32_t)p.M};
    const cuuint32_t elem[3] = {1, 1, 1};
    const CUtensorMapDataType dtype = sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    const CUresult r = encode(&tmap, dtype, 3, (void*)heat, dims, strides, box, elem, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return OKP_E_CUDA;
    const bool fused = ga != nullptr && sp.F > 0;
    auto kernel = fused ? okp_peaks_stream_kernel<T, true> : okp_peaks_stream_kernel<T, false>;
    OkpGroupArgs none;
    if (!fused) memset(&none, 0, sizeof(none));
    OKP_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, sp.smem_bytes));
    int per_sm = 0;
    OKP_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, sp.threads, sp.smem_bytes));
    if (per_sm < 1) return OKP_E_UNSUPPORTED;
    int device = 0, sms = 148;
    OKP_CUDA_CHECK(cudaGetDevice(&device));
    OKP_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    long long grid = (long long)per_sm * sms;               // persistent: every CTA resident, groups dealt round-robin
    if (grid > sp.groups) grid = sp.groups;
    const float thr_lo = threshold - OKP_STRIP_THRESHOLD_SLACK * fabsf(threshold);
    OKP_CUDA_CHECK(cudaMemsetAsync(group_counter_dev, 0, sizeof(int), stream));
    if (before) OKP_CUDA_CHECK(cudaEventRecord(before, stream));
    kernel<<<(unsigned)grid, sp.threads, sp.smem_bytes, stream>>>(tmap, heat, sp, threshold, thr_lo, tables, fused ? *ga : none,
                                                                  group_counter_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    if (after) OKP_CUDA_CHECK(cudaEventRecord(after, stream));
    return OKP_OK;
}
