// okp_peaks_strip.cuh -- tuned K1 for sm_100a: TMA-fed strip kernel, bounded filter + exact check.
//
// Replaces perception/pipeline.py:46-79 + perception/models.py:55-58 for every map of a batch.
//
// Why this shape. A peak is a pixel whose 5x5 box sum S (25 float32 additions in raster tap order,
// SURVEY.md section 7: torch's CPU conv2d is bitwise that) exceeds the threshold and equals the
// maximum of S over its 5x5 neighbourhood. Computing S exactly for every pixel costs 24
// dependent-order FADDs per pixel and made the first version of this kernel issue-bound at 0.31 of
// the HBM roofline (profiles/r01a_k1_strip_ncu.md). Peaks are rare, so the stream computes a cheap
// BOUND instead and the exact arithmetic runs only where the bound cannot decide:
//
//   * every pixel gets the separable sum S~ (horizontal 5-sums shared between the 4 pixels of a
//     strip, vertical 5-sum from running pair sums: 5.25 FADD per pixel). For non-negative inputs
//     any summation order of the same 25 terms is within gamma_24 * sum|x| of the true sum, so
//     |S - S~| <= 2.9e-6 * S~. With tie = 1 + 2e-5: S~(p) <= threshold * (1 - 1e-5) proves
//     S(p) <= threshold, and S~(q) > tie * S~(p) proves S(q) > S(p). Pixels that survive both tests
//     against the part of their neighbourhood the warp can see are CANDIDATES (true peaks, near
//     ties, and the odd pixel on a warp edge);
//   * a candidate carries a 25-bit mask of the neighbours the stream could not order (S~ inside
//     the tie band, or held by another warp). The epilogue computes the candidate's S exactly (25
//     loads from L2, raster-order __fadd_rn), compares it with the threshold, and with the exact S of
//     every masked neighbour (normally none). The peak set, the scores and the raster order are
//     therefore bit-identical to the exact kernel's; ties keep every tied pixel like `x == hmax`;
//   * maps holding a negative value void the bound, and so do NaN / Inf (torch's max_pool2d propagates NaN:
//     no pixel whose window holds a NaN box sum is a peak). The stream ORs the bits of every value
//     (2 LOP3 per row); bit 31 = a negative value, bit 30 = a value >= 2.0, an Inf or a NaN (probabilities
//     never set it). Such maps are handed to the exact generic kernels through the overflow path, like maps
//     with more than K peaks ("the first K in raster order").
//
// Data movement: heatmap rows arrive in shared memory by TMA (cp.async.bulk.tensor, one elected
// thread of a producer warp); the tensor map's out-of-bounds zero fill IS conv2d's zero padding.
// TMA wants the innermost start coordinate 16-byte aligned (tools/microbench/tma_probe.cu), so the
// box starts at column -4 and strip s produces the pixels x = 4s-2 .. 4s+1 from the columns
// 4s-4 .. 4s+3 = two aligned LDS.128. A thread owns one strip of one map and slides down it with
// everything in registers (running pair sums, the last five rows of S~); per row step: 2 LDS.128,
// 21 FADD, 3 FMNMX + 1 compare + 1 vote. The 5x5 maximum is formed from the strip's own column maxima
// and those of the two neighbouring lanes (4 shuffles, only in warps that hold a pixel above the
// threshold). Nothing is written in the row loop and the compute warps wait for nothing but the TMA
// barrier: the second version of this kernel (profiles/r01b_k1_ncu.md) kept S~ in a shared-memory
// ring that service warps tested, and spent 42 % of its issue slots in the mbarrier spin loops of
// that hand-over.
#pragma once
#include <cuda.h>

#include "okp_common.cuh"
#include "okp_peaks.cuh"

#define OKP_STRIP_RB 5            // rows per batch (= period of the register rings, so slots are static)
#define OKP_STRIP_MAX_NS 8        // TMA stages (upper bound; the plan picks NS)
#define OKP_STRIP_TIE 1.00002f    // S~(q) > tie * S~(p) proves S(q) > S(p)   (see the header)
#define OKP_STRIP_THRESHOLD_SLACK 1e-5f
#define OKP_STRIP_MAX_THREADS 640

struct OkpStripPlan {
    int H, W, maps;
    int strips;                   // W / 4 + 1 (strip s = pixels 4s-2 .. 4s+1)
    int half_strips;              // strips served by TMA box 0 (all of them when halves == 1)
    int halves;                   // 1 or 2 TMA boxes per row (box width <= 256 elements)
    int BW;                       // box width in elements
    int esize;                    // bytes per map element: 4 (float32) or 2 (bfloat16)
    int lead[2];                  // elements between a box's first column and its first strip's column 4s-4
                                  // (the box start must be 16-byte aligned: 0 for float32, 0 or 4 for bfloat16)
    int M;                        // maps per CTA
    int NS;                       // TMA stages
    int nb;                       // batches
    int K;                        // table capacity per map
    int PK;                       // candidate slots per map (2 K)
    int IC;                       // exact-check items per CTA (neighbours the stream could not order)
    int threads;                  // compute threads: M * strips (dense: a warp may hold strips of two maps)
    int half_bytes;               // bytes of one TMA box: M * RB * BW * esize
    int half_stride;              // half_bytes rounded up to 128 (TMA destinations are 128-byte aligned)
    int stage_bytes;              // halves * half_stride
};

struct OkpStripPeak { int32_t key; float score, cx, cy, conf; };   // key < 0: not a peak
struct OkpStripCandidate { int32_t key; uint32_t ties; };          // ties: bit k = neighbour (k / 5 - 2, k % 5 - 2) needs the exact check

__device__ __forceinline__ uint32_t okp_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void okp_mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(okp_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void okp_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(okp_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool okp_mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(okp_smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// try_wait with a suspend-time hint: the thread sleeps in hardware until the phase completes or the hint (in ns-scale
// ticks) runs out, instead of coming back after the short default time-out and spinning through the instruction issue
// slots of the warps that do the work (the producer's wait loop was 15 % of K1's executed instructions, r01v).
__device__ __forceinline__ bool okp_mbar_try_wait_suspend(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(okp_smem_u32(bar)), "r"(parity), "r"(0x989680u) : "memory");
    return ok != 0;
}
// Waits for the phase with the given parity. A wait that lasts longer than ~2 s of SM clocks can only
// be a protocol bug: trap (the launch fails with an error) instead of hanging the GPU. The loop is lean on purpose -- a
// waiting warp shares its scheduler with working ones: the clock is read once per 256 polls, and `pause_ns` is the sleep
// between polls (20 ns where the wait is on the critical path; the epilogue warps, which wait tens of microseconds for a
// group's candidates, pass a longer one).
__device__ __forceinline__ void okp_mbar_wait(uint64_t* bar, uint32_t parity, unsigned pause_ns = 20) {
    if (okp_mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    for (unsigned polls = 1;; ++polls) {
        if (okp_mbar_try_wait_suspend(bar, parity)) return;
        if ((polls & 255u) == 0u && clock64() - t0 > 4000000000LL) __trap();
        __nanosleep(pause_ns);
    }
}
__device__ __forceinline__ void okp_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(okp_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void okp_tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(okp_smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(okp_smem_u32(bar)) : "memory");
}


// The reference's box sum at pixel (y, x): 25 additions in raster tap order starting from +0, zero
// outside the image (perception/pipeline.py:70-71). The loads are independent (one L2 round trip).
template <typename T>
__device__ __forceinline__ float okp_exact_box_sum(const T* __restrict__ src, int H, int W, int y, int x) {
    float q[25];
#pragma unroll
    for (int k = 0; k < 25; ++k) {
        const int i2 = y + k / 5 - 2, j2 = x + k % 5 - 2;
        const bool in = i2 >= 0 && i2 < H && j2 >= 0 && j2 < W;
        q[k] = in ? okp_ld<T>(src + (size_t)i2 * W + j2) : 0.0f;
    }
    float acc = 0.0f;
#pragma unroll
    for (int k = 0; k < 25; ++k) acc = __fadd_rn(acc, q[k]);
    return acc;
}

// What a compute thread knows about its strip (loop invariant).
struct OkpStripLane {
    int H, W;
    float thr_lo;
    int xs;                        // 4 * strip: the strip's pixels are xs-2 .. xs+1
    uint32_t vmask;                // bit c: pixel xs+c-2 is inside the image; bit 4 / 5: lane-1 / lane+1 holds strip s-1 / s+1
    OkpStripCandidate* pending;    // this map's candidate list
    int* n_pending;
    int PK;
};

// One row step of the sliding window. I = step inside the batch = slot of the register rings.
// (lo, hi) are the columns 4s-4 .. 4s+3 of the new input row y + 2; the step produces S~ of row y for
// the strip's pixels x = xs + c - 2 (c = 0..3). pr keeps the running pair sums h(t-1) + h(t) of the
// horizontal sums, sv the strip's last five rows of S~, so that the pixels of row y - 2 can be tested
// against their 5x5 neighbourhood as soon as S~ of row y is known. EDGE = false: the batch lies in the
// interior of the map (every row of every neighbourhood exists), which saves the -inf padding selects.
template <int I, bool EDGE>
__device__ __forceinline__ void okp_strip_step(const float4 lo, const float4 hi, float (&pr)[5][4], float (&hp)[4],
                                               float (&sv)[5][4], uint32_t& sign, int y, const OkpStripLane& L) {
    // horizontal 5-sums of the four windows w[c .. c+4] (w = lo.xyzw, hi.xyzw): 9 adds
    const float c34 = lo.w + hi.x;
    const float t12 = lo.y + lo.z;
    const float t56 = hi.y + hi.z;
    const float tc = t12 + c34;
    const float u = c34 + t56;
    float h[4];
    h[0] = lo.x + tc; h[1] = tc + hi.y; h[2] = lo.z + u; h[3] = u + hi.w;
    // the strip's own pixels are w[2..5]: a set sign bit anywhere voids the bound (see the header)
    sign |= __float_as_uint(lo.z) | __float_as_uint(lo.w);
    sign |= __float_as_uint(hi.x) | __float_as_uint(hi.y);
    // vertical: S~(t) = P(t-3) + P(t-1) + h(t), P(t) = h(t-1) + h(t): 12 adds
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        sv[I][c] = (pr[(I + 2) % 5][c] + pr[(I + 4) % 5][c]) + h[c];
        pr[I][c] = hp[c] + h[c];
        hp[c] = h[c];
    }
    // ---- row yc = y - 2 (slot R2), whose five rows of S~ are now known ----
    const int yc = y - 2;
    if (EDGE && (yc < 0 || yc >= L.H)) return;                      // uniform over the CTA
    constexpr int R2 = (I + 3) % 5;
    const float (&b)[4] = sv[R2];
    // warp-uniform branch (taken by about a quarter of the warp rows of a busy map)
    if (!__any_sync(0xffffffffu, fmaxf(fmaxf(b[0], b[1]), fmaxf(b[2], b[3])) > L.thr_lo)) return;
    const float ninf = -INFINITY;
    const uint32_t vmask = L.vmask;
    const float tie = OKP_STRIP_TIE;
    // rows yc-2, yc-1 (slots I+1, I+2) and yc+1, yc+2 (slots I+4, I) may lie outside the image: max_pool2d pads with -inf
    const bool up2 = !EDGE || yc >= 2, up1 = !EDGE || yc >= 1, dn1 = !EDGE || yc + 1 < L.H, dn2 = !EDGE || yc + 2 < L.H;
    // second gate, still from registers only: a peak is at least a VERTICAL local maximum, so a row in which no pixel
    // above the threshold is (within the tie band) as large as the pixels right above and below it cannot hold a
    // candidate. A blob's box sum stays above the threshold over ~10 rows but has its vertical maximum in one or two
    // of them: this skips the 5x5 neighbourhood test (a third of the kernel's instructions, r01l) for nine busy rows in ten.
    {
        int possible = 0;                                         // bitwise on purpose: no short-circuit branches
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const float v = fmaxf(up1 ? sv[(I + 2) % 5][c] : ninf, dn1 ? sv[(I + 4) % 5][c] : ninf);
            possible |= (int)(b[c] > L.thr_lo) & (int)(b[c] * tie >= v);
        }
        if (!__any_sync(0xffffffffu, possible != 0)) return;
    }
    float own[4], cm[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        float m = fmaxf(up2 ? sv[(I + 1) % 5][c] : ninf, up1 ? sv[(I + 2) % 5][c] : ninf);
        m = fmaxf(m, fmaxf(dn1 ? sv[(I + 4) % 5][c] : ninf, dn2 ? sv[I][c] : ninf));
        own[c] = m;                                                  // column c without the centre row
        cm[c] = ((vmask >> c) & 1u) ? fmaxf(m, b[c]) : ninf;         // columns outside the image never win
    }
    // columns -2, -1 from the strip to the left, 4, 5 from the strip to the right. Where the neighbouring
    // lane does not hold that strip (warp edge: unknown; image edge: nothing there) -inf keeps the test
    // conservative and the unknown pixels go into the candidate's exact-check mask
    float l2 = __shfl_up_sync(0xffffffffu, cm[2], 1), l3 = __shfl_up_sync(0xffffffffu, cm[3], 1);
    float r0 = __shfl_down_sync(0xffffffffu, cm[0], 1), r1 = __shfl_down_sync(0xffffffffu, cm[1], 1);
    if (!(vmask & 16u)) { l2 = ninf; l3 = ninf; }
    if (!(vmask & 32u)) { r0 = ninf; r1 = ninf; }
    // maximum over the pixel's neighbours (5 columns x 5 rows without the pixel itself)
    const float q0 = fmaxf(fmaxf(l2, l3), fmaxf(cm[1], cm[2])), q3 = fmaxf(fmaxf(cm[1], cm[2]), fmaxf(r0, r1));
    const float others[4] = {fmaxf(own[0], q0), fmaxf(fmaxf(l3, cm[0]), fmaxf(own[1], fmaxf(cm[2], cm[3]))),
                             fmaxf(fmaxf(cm[0], cm[1]), fmaxf(own[2], fmaxf(cm[3], r0))), fmaxf(own[3], q3)};
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        // a candidate: above the threshold, inside the image, and no visible neighbour is provably larger
        if (!(b[c] > L.thr_lo && b[c] * tie >= others[c] && ((vmask >> c) & 1u))) continue;
        // neighbours that are not provably smaller go into the exact-check mask: all of them when any is inside the
        // tie band (rare), and the columns another warp holds; the epilogue drops the ones outside the image
        uint32_t ties = others[c] * tie >= b[c] ? 0x1FFEFFFu : 0u;
        if (c < 2 && !(vmask & 16u)) ties |= c == 0 ? 0x318C63u : 0x108421u;
        if (c > 1 && !(vmask & 32u)) ties |= c == 3 ? 0x18C6318u : 0x1084210u;
        const int entry = atomicAdd(L.n_pending, 1);
        if (entry < L.PK) {
            OkpStripCandidate cd;
            cd.key = yc * L.W + L.xs + c - 2;
            cd.ties = ties;
            L.pending[entry] = cd;
        }
    }
}

// The eight columns 4s-4 .. 4s+3 of one staged row as float32. float32 maps: two aligned LDS.128.
// bfloat16 maps: the window is 16 bytes at an 8-byte aligned address (two LDS.64); a bf16 is the upper
// half of the float32 with the same value, so the conversion is a shift / a mask per element (exact).
template <typename T> __device__ __forceinline__ void okp_strip_window(const unsigned char* row, float4& lo, float4& hi);
template <> __device__ __forceinline__ void okp_strip_window<float>(const unsigned char* row, float4& lo, float4& hi) {
    lo = reinterpret_cast<const float4*>(row)[0];
    hi = reinterpret_cast<const float4*>(row)[1];
}
template <> __device__ __forceinline__ void okp_strip_window<__nv_bfloat16>(const unsigned char* row, float4& lo, float4& hi) {
    const uint2 a = reinterpret_cast<const uint2*>(row)[0], b = reinterpret_cast<const uint2*>(row)[1];
    lo.x = __uint_as_float(a.x << 16); lo.y = __uint_as_float(a.x & 0xFFFF0000u);
    lo.z = __uint_as_float(a.y << 16); lo.w = __uint_as_float(a.y & 0xFFFF0000u);
    hi.x = __uint_as_float(b.x << 16); hi.y = __uint_as_float(b.x & 0xFFFF0000u);
    hi.z = __uint_as_float(b.y << 16); hi.w = __uint_as_float(b.y & 0xFFFF0000u);
}

// One batch of RB rows: the five unrolled steps, rows fetched one step ahead of their use (two register
// pairs, ping-pong). raw: this thread's window in the stage; y0: the batch's first output row.
template <bool EDGE, typename T>
__device__ __forceinline__ void okp_strip_batch(const unsigned char* raw, int row_pitch, float (&pr)[5][4], float (&hp)[4],
                                                float (&sv)[5][4], uint32_t& sign, int y0, const OkpStripLane& L) {
    float4 a0, a1, b0, b1;
    okp_strip_window<T>(raw, a0, a1);
    okp_strip_window<T>(raw + row_pitch, b0, b1);
    okp_strip_step<0, EDGE>(a0, a1, pr, hp, sv, sign, y0 + 0, L);
    okp_strip_window<T>(raw + 2 * row_pitch, a0, a1);
    okp_strip_step<1, EDGE>(b0, b1, pr, hp, sv, sign, y0 + 1, L);
    okp_strip_window<T>(raw + 3 * row_pitch, b0, b1);
    okp_strip_step<2, EDGE>(a0, a1, pr, hp, sv, sign, y0 + 2, L);
    okp_strip_window<T>(raw + 4 * row_pitch, a0, a1);
    okp_strip_step<3, EDGE>(b0, b1, pr, hp, sv, sign, y0 + 3, L);
    okp_strip_step<4, EDGE>(a0, a1, pr, hp, sv, sign, y0 + 4, L);
}

// ---------------------------------------------------------------------------------------------
// host side: tensor map encoder (the plan and the launch are in okp_peaks_stream.cuh)
// ---------------------------------------------------------------------------------------------
static inline int okp_round_up_int(int v, int m) { return (v + m - 1) / m * m; }

typedef CUresult (*OkpEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                     CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline OkpEncodeTiledFn okp_encode_tiled_fn() {
    static OkpEncodeTiledFn fn = nullptr;                 // resolved once; a function pointer is not library state
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult status;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &status) != cudaSuccess ||
            status != cudaDriverEntryPointSuccess)
            return nullptr;
        fn = (OkpEncodeTiledFn)ptr;
    }
    return fn;
}
