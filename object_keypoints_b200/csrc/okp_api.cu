// okp_api.cu -- the extern "C" surface of libokp.so (declared in include/okp.h): argument
// checking, launch planning, kernel launches. No allocation, no global state, no implicit sync.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "okp_common.cuh"
#include "okp_peaks.cuh"
#include "okp_peaks_strip.cuh"
#include "okp_peaks_stream.cuh"
#include "okp_geometry.cuh"
#include "okp_group.cuh"
#include "okp_dlt.cuh"
#include "okp_stereo.cuh"
#include "okp_sequence.cuh"
#include "okp_eval.cuh"
#include "okp_records.cuh"
#include "okp_targets.cuh"
#include "okp_sparse.cuh"

namespace {

constexpr int kSmCount = 148;            // B200: 2 dies x 74 SMs

struct PeakPlan {
    bool strip;                          // the stream kernel (plan sp) + overflow path, else generic tile kernel + merge
    OkpStreamPlan sp;                    // peaks only (sp.F = 0)
    OkpTileGeometry geo;                 // generic tiles (also the strip kernel's overflow path)
    size_t smem_bytes;
    int grid;
    int tiles_per_map;
};

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

PeakPlan plan_peaks(int maps, int C, int H, int W, int K, int esize, const OkpDecodeParams* prm) {
    PeakPlan p;
    memset(&p, 0, sizeof(p));
    // the stream kernel implements the reference's configuration only (5x5 window on the 5x5 box sum)
    const bool reference_mode = prm->nms_size == 5 && prm->box_sum == 1;
    p.strip = reference_mode && okp_stream_plan(maps, C, H, W, K, esize, 0, prm->lean_tables, &p.sp);
    p.geo.H = H; p.geo.W = W; p.geo.maps = maps;
    p.geo.radius = prm->nms_size / 2; p.geo.box_sum = prm->box_sum ? 1 : 0;
    p.geo.TW = W <= 64 ? round_up(W, 8) : 64;
    p.geo.TH = H <= 64 ? H : 32;
    p.geo.tiles_x = (W + p.geo.TW - 1) / p.geo.TW;
    p.geo.tiles_y = (H + p.geo.TH - 1) / p.geo.TH;
    p.smem_bytes = sizeof(float) * ((size_t)(p.geo.TH + 8) * (p.geo.TW + 8) + (size_t)(p.geo.TH + 4) * (p.geo.TW + 4)) +
                   sizeof(int32_t) * 2 * (size_t)K;
    p.tiles_per_map = p.geo.tiles_x * p.geo.tiles_y;
    const long long work = (long long)maps * p.tiles_per_map;
    const long long resident = (long long)kSmCount * 8;
    p.grid = (int)(work < resident ? work : resident);
    if (p.grid < 1) p.grid = 1;
    return p;
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int check_params(const OkpDecodeParams* prm) {
    if (!prm) return OKP_E_NULL;
    if (prm->max_peaks < 1 || prm->max_peaks > OKP_MAX_PEAKS) return OKP_E_CAPACITY;
    if (prm->max_objects < 1 || prm->max_objects > OKP_MAX_OBJECTS) return OKP_E_CAPACITY;
    if (prm->max_votes < 1 || prm->max_votes > 4096) return OKP_E_CAPACITY;
    if ((prm->nms_size != 5 && prm->nms_size != 3) || (prm->box_sum != 0 && prm->box_sum != 1)) return OKP_E_UNSUPPORTED;
    if (prm->top_k < 0 || prm->top_k > prm->max_peaks) return OKP_E_CAPACITY;
    if (prm->lean_tables != 0 && prm->lean_tables != 1) return OKP_E_UNSUPPORTED;
    if (prm->single_pass != 0 && prm->single_pass != 1) return OKP_E_UNSUPPORTED;
    return OKP_OK;
}

int check_shape(int N, int C, int H, int W) {
    if (N < 0 || C < 1 || C > OKP_MAX_MAPS || H < 1 || W < 1) return OKP_E_SHAPE;
    if ((long long)H * W > (1LL << 30)) return OKP_E_SHAPE;      // the raster key y * W + x is an int32
    return OKP_OK;
}

// CTAs of the overflow fix-up and the maps each of them owns (okp_peaks_overflow_kernel)
inline int overflow_grid(int maps) { return maps < OKP_OVERFLOW_CTAS ? maps : OKP_OVERFLOW_CTAS; }
inline int overflow_maps_per_cta(int maps) { return (maps + overflow_grid(maps) - 1) / overflow_grid(maps); }

// tile lists: one per (map, tile) for the generic kernels, one per (overflow CTA, tile) for the strip path
size_t workspace_for(const PeakPlan& p, int maps, int K) {
    const size_t tiles = p.strip ? (size_t)overflow_grid(maps) * p.tiles_per_map : (size_t)maps * p.tiles_per_map;
    // + alignment slack in front, + the launch's group counter (okp_peaks_stream.cuh) behind the lists
    return align_up(tiles * sizeof(int32_t), 256) + align_up(tiles * K * sizeof(OkpPeakRecord), 256) + 256 + 256;
}

}  // namespace

extern "C" {

int okp_version(void) { return OKP_VERSION_MAJOR * 1000 + OKP_VERSION_MINOR; }

const char* okp_strerror(int code) {
    switch (code) {
        case OKP_OK: return "ok";
        case OKP_E_NULL: return "a required pointer is NULL";
        case OKP_E_SHAPE: return "shape out of the supported range";
        case OKP_E_CAPACITY: return "max_peaks / max_objects / max_votes out of range";
        case OKP_E_UNSUPPORTED: return "parameter combination not implemented";
        case OKP_E_CUDA: return "CUDA runtime call or kernel launch failed";
        case OKP_E_WORKSPACE: return "workspace too small (see okp_decode_workspace_bytes)";
        default: return "unknown error code";
    }
}

size_t okp_decode_workspace_bytes(int N, int C, int H, int W, const OkpDecodeParams* params) {
    if (check_params(params) != OKP_OK || check_shape(N, C, H, W) != OKP_OK) return 0;
    if (N == 0) return 256;
    // enough for every element type (their launch plans can differ: 16-bit rows need W % 8 == 0 for TMA; bf16 and f16
    // share one plan)
    size_t need = 0;
    for (int esize = 2; esize <= 4; esize += 2) {
        const PeakPlan p = plan_peaks(N * C, C, H, W, params->max_peaks, esize, params);
        const size_t bytes = workspace_for(p, N * C, params->max_peaks);
        if (bytes > need) need = bytes;
    }
    return need;
}

}  // extern "C"

namespace {

// Everything the peak entry checks before it launches; fills the plan and the workspace carving.
struct PeakCall {
    PeakPlan plan;
    int32_t* tile_count;
    OkpPeakRecord* tile_peaks;
    int* group_counter;                  // one int the stream kernel's CTAs claim their groups from
};

template <typename T>
int prepare_peaks(const T* heat_dev, int N, int C, int H, int W, const OkpDecodeParams* params,
                  const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes, PeakCall* call) {
    if (!heat_dev || !tables || !workspace_dev) return OKP_E_NULL;
    if (!tables->peak_count || !tables->peak_yx || !tables->peak_score || !tables->peak_xy || !tables->peak_conf ||
        !tables->peak_object || !tables->peak_vote)
        return OKP_E_NULL;
    // the table writers use 8- and 16-byte vector stores (int2 / float2 / double2 rows)
    if (((uintptr_t)tables->peak_yx & 7u) || ((uintptr_t)tables->peak_xy & 7u) || ((uintptr_t)tables->peak_vote & 15u))
        return OKP_E_UNSUPPORTED;
    const int K = params->max_peaks;
    const int maps = N * C;
    call->plan = plan_peaks(maps, C, H, W, K, (int)sizeof(T), params);
    // TMA needs a 16-byte aligned base. The generic kernels would take the map, but with a workspace orders of magnitude
    // larger than okp_decode_workspace_bytes() advertises for this shape: refuse instead of failing later
    if (call->plan.strip && ((uintptr_t)heat_dev & 15u) != 0) return OKP_E_UNSUPPORTED;
    if (workspace_bytes < workspace_for(call->plan, maps, K)) return OKP_E_WORKSPACE;
    const size_t tiles = call->plan.strip ? (size_t)overflow_grid(maps) * call->plan.tiles_per_map : (size_t)maps * call->plan.tiles_per_map;
    uintptr_t base = align_up((uintptr_t)workspace_dev, 256);
    call->tile_count = (int32_t*)base;
    call->tile_peaks = (OkpPeakRecord*)(base + align_up(tiles * sizeof(int32_t), 256));
    call->group_counter = (int*)((uintptr_t)call->tile_peaks + align_up(tiles * K * sizeof(OkpPeakRecord), 256));
    return OKP_OK;
}

// maps with more than K peaks ("first K in raster order"), negative / NaN values ... are redone here; a no-op otherwise
template <typename T>
int launch_overflow(const T* heat_dev, const PeakCall& call, int maps, const OkpDecodeParams* params,
                    const OkpDecodeTables* tables, cudaStream_t s) {
    auto kernel = okp_peaks_overflow_kernel<256, T>;
    OKP_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)call.plan.smem_bytes));
    OKP_CUDA_CHECK(okp_launch_dependent(kernel, dim3(overflow_grid(maps)), dim3(256), call.plan.smem_bytes, s, heat_dev, call.plan.geo,
                                        params->threshold, params->max_peaks, overflow_maps_per_cta(maps), call.tile_count,
                                        call.tile_peaks, *tables));
    return OKP_OK;
}

// The peak extraction's launches for a prepared call: the stream kernel + overflow fix-up, or the generic kernels + merge.
template <typename T>
int launch_peaks(const T* heat_dev, const PeakCall& call, int maps, int C, int W, const OkpDecodeParams* params,
                 const OkpDecodeTables* tables, cudaStream_t s, void* event_before = nullptr, void* event_after = nullptr) {
    const int K = params->max_peaks;
    const PeakPlan& p = call.plan;
    if (p.strip) {
        int rc = okp_stream_launch<T>(heat_dev, p.sp, params->threshold, *tables, nullptr, call.group_counter, s,
                                      (cudaEvent_t)event_before, (cudaEvent_t)event_after);
        if (rc != OKP_OK) return rc;
        rc = launch_overflow<T>(heat_dev, call, maps, params, tables, s);
        if (rc != OKP_OK) return rc;
    } else {
        auto kernel = okp_peaks_generic_kernel<256, T>;
        OKP_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_bytes));
        kernel<<<p.grid, 256, p.smem_bytes, s>>>(heat_dev, p.geo, params->threshold, K, call.tile_count, call.tile_peaks);
        OKP_CUDA_CHECK(cudaGetLastError());
        const int warps_per_block = 4;
        okp_merge_peaks_kernel<<<(maps + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, s>>>(
            call.tile_count, call.tile_peaks, maps, p.tiles_per_map, W, K, C, *tables);
        OKP_CUDA_CHECK(cudaGetLastError());
    }
    if (params->top_k > 0) {
        okp_topk_kernel<<<(maps + 3) / 4, 128, 0, s>>>(maps, K, params->top_k, *tables);
        OKP_CUDA_CHECK(cudaGetLastError());
    }
    return OKP_OK;
}

template <typename T>
int extract_peaks(const T* heat_dev, int N, int C, int H, int W, const OkpDecodeParams* params,
                  const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes, void* stream,
                  void* event_before = nullptr, void* event_after = nullptr) {
    int rc = check_params(params);
    if (rc != OKP_OK) return rc;
    rc = check_shape(N, C, H, W);
    if (rc != OKP_OK) return rc;
    if (N == 0) return OKP_OK;
    PeakCall call;
    rc = prepare_peaks<T>(heat_dev, N, C, H, W, params, tables, workspace_dev, workspace_bytes, &call);
    if (rc != OKP_OK) return rc;
    return launch_peaks<T>(heat_dev, call, N * C, C, W, params, tables, (cudaStream_t)stream, event_before, event_after);
}

int convert_sink(const OkpRecordSink* sink, int O, int C, int P, OkpRecordSinks* out) {
    memset(out, 0, sizeof(*out));
    if (!sink || sink->n_buffers == 0) return OKP_OK;
    if (sink->n_buffers < 0 || sink->n_buffers > OKP_MAX_PEERS || sink->first_row < 0) return OKP_E_SHAPE;
    if (sink->record_bytes < okp_compact_record_bytes(O, C, P) || (sink->record_bytes & 7)) return OKP_E_SHAPE;
    if (!sink->buffers_dev) return OKP_E_NULL;
    for (int d = 0; d < sink->n_buffers; ++d) {
        if (!sink->buffers_dev[d]) return OKP_E_NULL;
        if ((uintptr_t)sink->buffers_dev[d] & 7u) return OKP_E_UNSUPPORTED;
        out->base[d] = (unsigned char*)sink->buffers_dev[d];
    }
    out->n = sink->n_buffers;
    out->stride = sink->record_bytes;
    out->first_row = sink->first_row;
    out->points_offset = okp_compact_points_offset(O, C);
    return OKP_OK;
}

// Checks and packs what the grouping needs (okp_group.cuh); *warps = frames per CTA of the stand-alone kernel.
// cameras_dev != NULL: the per-frame-camera form (okp_group_cameras_kernel), whose scratch also holds the frame's camera.
int make_group_args(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                    const int32_t* keypoint_config, const OkpCamera* camera, const OkpCamera* cameras_dev,
                    const OkpDecodeParams* params, const OkpDecodeTables* tables, const OkpRecordSink* sink, OkpGroupArgs* a) {
    if (!tables || (C > 1 && (!centers_dev || !keypoint_config))) return OKP_E_NULL;
    if ((camera || cameras_dev) && !depth_dev) return OKP_E_NULL;
    const void* const* fields = (const void* const*)tables;
    for (size_t i = 0; i < sizeof(OkpDecodeTables) / sizeof(void*); ++i)
        if (!fields[i]) return OKP_E_NULL;
    // vector stores: double2 rows of peak_vote / votes, float2 rows of kp_xy
    if (((uintptr_t)tables->peak_vote & 15u) || ((uintptr_t)tables->votes & 15u) || ((uintptr_t)tables->kp_xy & 7u) ||
        ((uintptr_t)tables->peak_xy & 7u))
        return OKP_E_UNSUPPORTED;
    memset(a, 0, sizeof(*a));
    a->config.cfg[0] = 1;                               // pipeline.py:36: centre map first
    int S = 1, P = 1;
    for (int i = 0; i < C - 1; ++i) {
        if (keypoint_config[i] < 1 || keypoint_config[i] > OKP_MAX_SLOTS) return OKP_E_CAPACITY;
        a->config.cfg[1 + i] = keypoint_config[i];
        if (keypoint_config[i] > S) S = keypoint_config[i];
        P += keypoint_config[i];
    }
    if (camera) a->cam = *camera;
    a->prm = *params;
    a->depth = depth_dev; a->centers = centers_dev;
    a->N = N; a->C = C; a->H = H; a->W = W; a->S = S; a->P = P;
    a->have_camera = camera != nullptr || cameras_dev != nullptr;
    const int K = params->max_peaks, O = params->max_objects;
    const size_t per_frame = okp_group_smem_bytes(C, K, O, cameras_dev != nullptr);
    if (per_frame > 200 * 1024) return OKP_E_CAPACITY;
    a->frame_smem_bytes = (int)per_frame;
    return convert_sink(sink, O, C, P, &a->sinks);
}

template <typename T, int LANES>
int launch_group_lanes(const OkpGroupArgs& a, int only_pending, const OkpDecodeTables* tables, const OkpCamera* cameras_dev,
                       cudaStream_t s) {
    const int most = 128 / LANES;                                          // frames per CTA: LANES lanes each
    int frames = (int)((size_t)(48 * 1024) / a.frame_smem_bytes);
    if (frames > most) frames = most;
    if (LANES == 16) frames &= ~1;                                         // whole warps (the caller checked that two frames fit)
    if (frames < 1) frames = 1;
    const size_t smem = (size_t)a.frame_smem_bytes * frames;
    const dim3 grid((a.N + frames - 1) / frames), block(frames * LANES);
    if (cameras_dev) {
        auto kernel = okp_group_cameras_kernel<T, LANES>;
        if (smem > 48 * 1024) OKP_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        OKP_CUDA_CHECK(okp_launch_dependent(kernel, grid, block, smem, s, a, *tables, cameras_dev));
        return OKP_OK;
    }
    auto kernel = okp_group_kernel<T, LANES>;
    if (smem > 48 * 1024) OKP_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    OKP_CUDA_CHECK(okp_launch_dependent(kernel, grid, block, smem, s, a, only_pending, *tables));
    return OKP_OK;
}

// Small frames hold few peaks (a 64x64 valve frame: ~10): half a warp per frame, two frames per warp (okp_group.cuh).
template <typename T>
int launch_group(const OkpGroupArgs& a, int only_pending, const OkpDecodeTables* tables, const OkpCamera* cameras_dev,
                 cudaStream_t s) {
    const bool small = (long long)a.H * a.W <= 96LL * 96LL && 2 * (size_t)a.frame_smem_bytes <= 48 * 1024;
    return small ? launch_group_lanes<T, 16>(a, only_pending, tables, cameras_dev, s)
                 : launch_group_lanes<T, 32>(a, only_pending, tables, cameras_dev, s);
}

// What the okp_*_cameras_* entries refuse on top of the checks of their single-camera twins. N <= 0 is left to those
// checks: like every entry, a call with no frames returns OKP_OK (an empty table may be NULL) and N < 0 is OKP_E_SHAPE.
int check_cameras(int N, const void* depth_dev, const OkpCamera* cameras_dev, const OkpDecodeParams* params) {
    if (N <= 0) return OKP_OK;
    if (!params || !cameras_dev || !depth_dev) return OKP_E_NULL;
    if ((uintptr_t)cameras_dev & 15u) return OKP_E_UNSUPPORTED;       // each lane copies one 16-byte word of the camera
    if (params->single_pass) return OKP_E_UNSUPPORTED;                // the fused single pass has no per-frame-camera form
    return OKP_OK;
}

// cameras_dev: NULL for the single-camera entries (camera, which may be NULL too, is the call's camera), else the
// per-frame camera table of okp_group_objects_cameras_* (camera NULL).
template <typename T>
int group_objects(const T* depth_dev, const T* centers_dev, int N, int C, int H, int W,
                  const int32_t* keypoint_config, const OkpCamera* camera, const OkpCamera* cameras_dev,
                  const OkpDecodeParams* params, const OkpDecodeTables* tables, const OkpRecordSink* sink, void* stream) {
    int rc = check_params(params);
    if (rc != OKP_OK) return rc;
    rc = check_shape(N, C, H, W);
    if (rc != OKP_OK) return rc;
    if (N == 0) return OKP_OK;
    OkpGroupArgs a;
    rc = make_group_args(depth_dev, centers_dev, N, C, H, W, keypoint_config, camera, cameras_dev, params, tables, sink, &a);
    if (rc != OKP_OK) return rc;
    return launch_group<T>(a, 0, tables, cameras_dev, (cudaStream_t)stream);
}

// ObjectKeypointPipeline.__call__ for a batch (perception/pipeline.py:182-200): the fused streaming pass where the
// shape and the mode allow it, else peak extraction followed by grouping.
template <typename T>
int decode(const T* heat_dev, const T* depth_dev, const T* centers_dev, int N, int C, int H, int W,
           const int32_t* keypoint_config, const OkpCamera* camera, const OkpCamera* cameras_dev, const OkpDecodeParams* params,
           const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes, const OkpRecordSink* sink,
           void* stream) {
    int rc = check_params(params);
    if (rc != OKP_OK) return rc;
    rc = check_shape(N, C, H, W);
    if (rc != OKP_OK) return rc;
    if (N == 0) return OKP_OK;
    OkpGroupArgs a;
    rc = make_group_args(depth_dev, centers_dev, N, C, H, W, keypoint_config, camera, cameras_dev, params, tables, sink, &a);
    if (rc != OKP_OK) return rc;
    PeakCall call;
    rc = prepare_peaks<T>(heat_dev, N, C, H, W, params, tables, workspace_dev, workspace_bytes, &call);
    if (rc != OKP_OK) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    // One fused pass (grouping in the peak kernel's epilogue warps) or two launches (peaks, then one warp per frame): the
    // grouping is a chain of latencies (gathers from HBM, float64 Newton + tan), and a launch of its own overlaps thousands
    // of them where the fused form has two epilogue warps per SM. Measured (profiles/r02c_fused_vs_split.txt): the split
    // form is faster at every size, so it is the default; OkpDecodeParams.single_pass asks for the fused one, whose groups
    // are whole frames with their grouping scratch: a plan of its own.
    OkpStreamPlan fused_plan;
    const bool fused = params->single_pass != 0 && !cameras_dev && call.plan.strip && params->top_k == 0 &&
                       okp_stream_plan(N * C, C, H, W, params->max_peaks, (int)sizeof(T), a.frame_smem_bytes, params->lean_tables,
                                       &fused_plan) && fused_plan.F > 0;
    if (!fused) {
        rc = launch_peaks<T>(heat_dev, call, N * C, C, W, params, tables, s);
        if (rc != OKP_OK) return rc;
        return launch_group<T>(a, 0, tables, cameras_dev, s);
    }
    rc = okp_stream_launch<T>(heat_dev, fused_plan, params->threshold, *tables, &a, call.group_counter, s);
    if (rc != OKP_OK) return rc;
    // fix-up launches: maps that overflowed the fast path are redone exactly, then their frames are grouped. With no such
    // map each is one read of peak_count / n_objects
    rc = launch_overflow<T>(heat_dev, call, N * C, params, tables, s);
    if (rc != OKP_OK) return rc;
    return launch_group<T>(a, 1, tables, nullptr, s);
}

}  // namespace

extern "C" {

int okp_extract_peaks_f32(const float* heat_dev, int N, int C, int H, int W, const OkpDecodeParams* params,
                          const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes, void* stream) {
    return extract_peaks<float>(heat_dev, N, C, H, W, params, tables, workspace_dev, workspace_bytes, stream);
}

int okp_extract_peaks_events_f32(const float* heat_dev, int N, int C, int H, int W, const OkpDecodeParams* params,
                                 const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes, void* event_before,
                                 void* event_after, void* stream) {
    return extract_peaks<float>(heat_dev, N, C, H, W, params, tables, workspace_dev, workspace_bytes, stream, event_before, event_after);
}

int okp_extract_peaks_bf16(const void* heat_dev, int N, int C, int H, int W, const OkpDecodeParams* params,
                           const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes, void* stream) {
    return extract_peaks<__nv_bfloat16>((const __nv_bfloat16*)heat_dev, N, C, H, W, params, tables, workspace_dev,
                                        workspace_bytes, stream);
}

int okp_extract_peaks_f16(const void* heat_dev, int N, int C, int H, int W, const OkpDecodeParams* params,
                          const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes, void* stream) {
    return extract_peaks<__half>((const __half*)heat_dev, N, C, H, W, params, tables, workspace_dev, workspace_bytes, stream);
}

int okp_group_objects_f32(const float* depth_dev, const float* centers_dev, int N, int C, int H, int W,
                          const int32_t* keypoint_config, const OkpCamera* camera, const OkpDecodeParams* params,
                          const OkpDecodeTables* tables, void* stream) {
    return group_objects<float>(depth_dev, centers_dev, N, C, H, W, keypoint_config, camera, nullptr, params, tables, nullptr, stream);
}

int okp_group_objects_bf16(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                           const int32_t* keypoint_config, const OkpCamera* camera, const OkpDecodeParams* params,
                           const OkpDecodeTables* tables, void* stream) {
    return group_objects<__nv_bfloat16>((const __nv_bfloat16*)depth_dev, (const __nv_bfloat16*)centers_dev, N, C, H, W,
                                        keypoint_config, camera, nullptr, params, tables, nullptr, stream);
}

int okp_group_objects_f16(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                          const int32_t* keypoint_config, const OkpCamera* camera, const OkpDecodeParams* params,
                          const OkpDecodeTables* tables, void* stream) {
    return group_objects<__half>((const __half*)depth_dev, (const __half*)centers_dev, N, C, H, W, keypoint_config, camera, nullptr,
                                 params, tables, nullptr, stream);
}

int okp_host_alias(const void* host_ptr, void** dev_ptr_out) {
    if (!host_ptr || !dev_ptr_out) return OKP_E_NULL;
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, host_ptr) != cudaSuccess) {
        cudaGetLastError();
        return OKP_E_UNSUPPORTED;
    }
    if (attr.type != cudaMemoryTypeHost || !attr.devicePointer) return OKP_E_UNSUPPORTED;
    *dev_ptr_out = attr.devicePointer;
    return OKP_OK;
}

int okp_decode_f32(const float* heat_dev, const float* depth_dev, const float* centers_dev, int N, int C, int H, int W,
                   const int32_t* keypoint_config, const OkpCamera* camera, const OkpDecodeParams* params,
                   const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes, void* stream) {
    return decode<float>(heat_dev, depth_dev, centers_dev, N, C, H, W, keypoint_config, camera, nullptr, params, tables, workspace_dev,
                         workspace_bytes, nullptr, stream);
}

int okp_decode_bf16(const void* heat_dev, const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                    const int32_t* keypoint_config, const OkpCamera* camera, const OkpDecodeParams* params,
                    const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes, void* stream) {
    return decode<__nv_bfloat16>((const __nv_bfloat16*)heat_dev, (const __nv_bfloat16*)depth_dev, (const __nv_bfloat16*)centers_dev,
                                 N, C, H, W, keypoint_config, camera, nullptr, params, tables, workspace_dev, workspace_bytes, nullptr, stream);
}

int okp_decode_f16(const void* heat_dev, const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                   const int32_t* keypoint_config, const OkpCamera* camera, const OkpDecodeParams* params,
                   const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes, void* stream) {
    return decode<__half>((const __half*)heat_dev, (const __half*)depth_dev, (const __half*)centers_dev, N, C, H, W,
                          keypoint_config, camera, nullptr, params, tables, workspace_dev, workspace_bytes, nullptr, stream);
}

int okp_record_bytes(int O, int C, const int32_t* keypoint_config) {
    if (O < 1 || O > OKP_MAX_OBJECTS || C < 1 || C > OKP_MAX_MAPS || (C > 1 && !keypoint_config)) return 0;
    int P = 1;
    for (int i = 0; i < C - 1; ++i) {
        if (keypoint_config[i] < 1 || keypoint_config[i] > OKP_MAX_SLOTS) return 0;
        P += keypoint_config[i];
    }
    return okp_compact_record_bytes(O, C, P);
}

int okp_decode_emit_f32(const float* heat_dev, const float* depth_dev, const float* centers_dev, int N, int C, int H, int W,
                        const int32_t* keypoint_config, const OkpCamera* camera, const OkpDecodeParams* params,
                        const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes,
                        const OkpRecordSink* sink, void* stream) {
    return decode<float>(heat_dev, depth_dev, centers_dev, N, C, H, W, keypoint_config, camera, nullptr, params, tables, workspace_dev,
                         workspace_bytes, sink, stream);
}

int okp_decode_emit_bf16(const void* heat_dev, const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                         const int32_t* keypoint_config, const OkpCamera* camera, const OkpDecodeParams* params,
                         const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes,
                         const OkpRecordSink* sink, void* stream) {
    return decode<__nv_bfloat16>((const __nv_bfloat16*)heat_dev, (const __nv_bfloat16*)depth_dev, (const __nv_bfloat16*)centers_dev,
                                 N, C, H, W, keypoint_config, camera, nullptr, params, tables, workspace_dev, workspace_bytes, sink, stream);
}

int okp_decode_emit_f16(const void* heat_dev, const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                        const int32_t* keypoint_config, const OkpCamera* camera, const OkpDecodeParams* params,
                        const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes,
                        const OkpRecordSink* sink, void* stream) {
    return decode<__half>((const __half*)heat_dev, (const __half*)depth_dev, (const __half*)centers_dev, N, C, H, W,
                          keypoint_config, camera, nullptr, params, tables, workspace_dev, workspace_bytes, sink, stream);
}

int okp_group_objects_emit_f32(const float* depth_dev, const float* centers_dev, int N, int C, int H, int W,
                               const int32_t* keypoint_config, const OkpCamera* camera, const OkpDecodeParams* params,
                               const OkpDecodeTables* tables, const OkpRecordSink* sink, void* stream) {
    return group_objects<float>(depth_dev, centers_dev, N, C, H, W, keypoint_config, camera, nullptr, params, tables, sink, stream);
}

int okp_group_objects_emit_bf16(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                                const int32_t* keypoint_config, const OkpCamera* camera, const OkpDecodeParams* params,
                                const OkpDecodeTables* tables, const OkpRecordSink* sink, void* stream) {
    return group_objects<__nv_bfloat16>((const __nv_bfloat16*)depth_dev, (const __nv_bfloat16*)centers_dev, N, C, H, W,
                                        keypoint_config, camera, nullptr, params, tables, sink, stream);
}

int okp_group_objects_emit_f16(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                               const int32_t* keypoint_config, const OkpCamera* camera, const OkpDecodeParams* params,
                               const OkpDecodeTables* tables, const OkpRecordSink* sink, void* stream) {
    return group_objects<__half>((const __half*)depth_dev, (const __half*)centers_dev, N, C, H, W, keypoint_config, camera, nullptr,
                                 params, tables, sink, stream);
}

int okp_decode_cameras_f32(const float* heat_dev, const float* depth_dev, const float* centers_dev, int N, int C, int H, int W,
                           const int32_t* keypoint_config, const OkpCamera* cameras_dev, const OkpDecodeParams* params,
                           const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes,
                           const OkpRecordSink* sink, void* stream) {
    const int rc = check_cameras(N, depth_dev, cameras_dev, params);
    if (rc != OKP_OK) return rc;
    return decode<float>(heat_dev, depth_dev, centers_dev, N, C, H, W, keypoint_config, nullptr, cameras_dev, params, tables,
                         workspace_dev, workspace_bytes, sink, stream);
}

int okp_decode_cameras_bf16(const void* heat_dev, const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                            const int32_t* keypoint_config, const OkpCamera* cameras_dev, const OkpDecodeParams* params,
                            const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes,
                            const OkpRecordSink* sink, void* stream) {
    const int rc = check_cameras(N, depth_dev, cameras_dev, params);
    if (rc != OKP_OK) return rc;
    return decode<__nv_bfloat16>((const __nv_bfloat16*)heat_dev, (const __nv_bfloat16*)depth_dev, (const __nv_bfloat16*)centers_dev,
                                 N, C, H, W, keypoint_config, nullptr, cameras_dev, params, tables, workspace_dev, workspace_bytes,
                                 sink, stream);
}

int okp_decode_cameras_f16(const void* heat_dev, const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                           const int32_t* keypoint_config, const OkpCamera* cameras_dev, const OkpDecodeParams* params,
                           const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes,
                           const OkpRecordSink* sink, void* stream) {
    const int rc = check_cameras(N, depth_dev, cameras_dev, params);
    if (rc != OKP_OK) return rc;
    return decode<__half>((const __half*)heat_dev, (const __half*)depth_dev, (const __half*)centers_dev, N, C, H, W,
                          keypoint_config, nullptr, cameras_dev, params, tables, workspace_dev, workspace_bytes, sink, stream);
}

int okp_group_objects_cameras_f32(const float* depth_dev, const float* centers_dev, int N, int C, int H, int W,
                                  const int32_t* keypoint_config, const OkpCamera* cameras_dev, const OkpDecodeParams* params,
                                  const OkpDecodeTables* tables, const OkpRecordSink* sink, void* stream) {
    const int rc = check_cameras(N, depth_dev, cameras_dev, params);
    if (rc != OKP_OK) return rc;
    return group_objects<float>(depth_dev, centers_dev, N, C, H, W, keypoint_config, nullptr, cameras_dev, params, tables, sink,
                                stream);
}

int okp_group_objects_cameras_bf16(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                                   const int32_t* keypoint_config, const OkpCamera* cameras_dev, const OkpDecodeParams* params,
                                   const OkpDecodeTables* tables, const OkpRecordSink* sink, void* stream) {
    const int rc = check_cameras(N, depth_dev, cameras_dev, params);
    if (rc != OKP_OK) return rc;
    return group_objects<__nv_bfloat16>((const __nv_bfloat16*)depth_dev, (const __nv_bfloat16*)centers_dev, N, C, H, W,
                                        keypoint_config, nullptr, cameras_dev, params, tables, sink, stream);
}

int okp_group_objects_cameras_f16(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                                  const int32_t* keypoint_config, const OkpCamera* cameras_dev, const OkpDecodeParams* params,
                                  const OkpDecodeTables* tables, const OkpRecordSink* sink, void* stream) {
    const int rc = check_cameras(N, depth_dev, cameras_dev, params);
    if (rc != OKP_OK) return rc;
    return group_objects<__half>((const __half*)depth_dev, (const __half*)centers_dev, N, C, H, W, keypoint_config, nullptr,
                                 cameras_dev, params, tables, sink, stream);
}

int okp_fisheye_undistort_f64(const double* xy_dev, int n, const OkpCamera* camera, int round_to_f32,
                              double* out_dev, void* stream) {
    if (n < 0) return OKP_E_SHAPE;
    if (n == 0) return OKP_OK;
    if (!xy_dev || !camera || !out_dev) return OKP_E_NULL;
    okp_undistort_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(xy_dev, n, *camera, round_to_f32, out_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_fisheye_project_f64(const double* X_dev, int n, const double* T_CW, const OkpCamera* camera, double* out_dev,
                            void* stream) {
    if (n < 0) return OKP_E_SHAPE;
    if (n == 0) return OKP_OK;
    if (!X_dev || !T_CW || !camera || !out_dev) return OKP_E_NULL;
    OkpPose pose;
    for (int i = 0; i < 12; ++i) pose.m[i] = T_CW[i];
    okp_project_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(X_dev, n, pose, *camera, out_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_detection_to_point_f32(const float* xy_dev, int n, const float* depth_map_dev, int H, int W,
                               const OkpCamera* camera, const OkpDecodeParams* params, double* out_dev, void* stream) {
    if (n < 0 || H < 1 || W < 1) return OKP_E_SHAPE;
    if (n == 0) return OKP_OK;
    if (!xy_dev || !depth_map_dev || !camera || !params || !out_dev) return OKP_E_NULL;
    okp_detection_to_point_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        xy_dev, n, depth_map_dev, H, W, *camera, params->compat_clip_bug, out_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_triangulate_f64(const double* points_dev, const uint8_t* valid_dev, const double* projections_dev,
                        int per_point_projections, int P, int V, double* out_dev, void* stream) {
    if (P < 0 || V < 1 || V > OKP_MAX_VIEWS) return OKP_E_SHAPE;
    if (P == 0) return OKP_OK;
    if (!points_dev || !projections_dev || !out_dev) return OKP_E_NULL;
    const size_t smem = per_point_projections ? 0 : sizeof(double) * 12 * (size_t)V;
    okp_triangulate_kernel<<<(P + 127) / 128, 128, smem, (cudaStream_t)stream>>>(
        points_dev, valid_dev, projections_dev, per_point_projections, P, V, out_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_reprojection_filter_f64(const double* X_dev, const double* obs_dev, uint8_t* valid_dev, const double* poses_dev,
                                const OkpCamera* camera, int P, int V, double max_error_px, double* err_dev,
                                void* stream) {
    if (P < 0 || V < 1 || V > OKP_MAX_VIEWS) return OKP_E_SHAPE;
    if (P == 0) return OKP_OK;
    if (!X_dev || !obs_dev || !valid_dev || !poses_dev || !camera || !err_dev) return OKP_E_NULL;
    const long long total = (long long)P * V;
    okp_reprojection_filter_kernel<<<(unsigned)((total + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        X_dev, obs_dev, valid_dev, poses_dev, *camera, P, V, max_error_px, err_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_triangulate_robust_f64(const double* obs_dev, uint8_t* valid_dev, const double* poses_dev,
                               const OkpCamera* camera, int P, int V, double max_error_px, int max_rounds,
                               double* out_dev, double* err_dev, int32_t* dropped_dev, void* stream) {
    if (P < 0 || V < 1 || V > OKP_MAX_VIEWS || max_rounds < 0) return OKP_E_SHAPE;
    if (P == 0) return OKP_OK;
    if (!obs_dev || !poses_dev || !camera || !out_dev || !err_dev) return OKP_E_NULL;
    const size_t smem = sizeof(double) * 24 * (size_t)V;
    okp_triangulate_robust_kernel<<<(P + 127) / 128, 128, smem, (cudaStream_t)stream>>>(
        obs_dev, valid_dev, poses_dev, *camera, P, V, max_error_px, max_rounds, out_dev, err_dev, dropped_dev, 0);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_triangulate_tracks_f64(const double* obs_dev, uint8_t* valid_dev, const double* poses_dev,
                               const OkpCamera* camera, int G, int Pg, int V, double max_error_px, int max_rounds,
                               double* out_dev, double* err_dev, int32_t* dropped_dev, void* stream) {
    if (G < 0 || Pg < 1 || V < 1 || V > OKP_MAX_VIEWS || max_rounds < 0 || G > 65535) return OKP_E_SHAPE;
    if ((long long)G * Pg > 0x7fffffffLL) return OKP_E_SHAPE;
    if (G == 0) return OKP_OK;
    if (!obs_dev || !poses_dev || !camera || !out_dev || !err_dev) return OKP_E_NULL;
    const size_t smem = sizeof(double) * 24 * (size_t)V;
    const int threads = Pg < 128 ? (Pg + 31) / 32 * 32 : 128;
    okp_triangulate_robust_kernel<<<dim3((Pg + threads - 1) / threads, G), threads, smem, (cudaStream_t)stream>>>(
        obs_dev, valid_dev, poses_dev, *camera, G * Pg, V, max_error_px, max_rounds, out_dev, err_dev, dropped_dev, Pg);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_correct_matches_f64(const double* F, const double* left_dev, const double* right_dev, int n, int round_to_f32,
                            double* left_out_dev, double* right_out_dev, void* stream) {
    if (n < 0) return OKP_E_SHAPE;
    if (n == 0) return OKP_OK;
    if (!F || !left_dev || !right_dev || !left_out_dev || !right_out_dev) return OKP_E_NULL;
    OkpMat3 Fm;
    for (int i = 0; i < 9; ++i) Fm.m[i] = F[i];
    okp_correct_matches_kernel<<<(n + 63) / 64, 64, 0, (cudaStream_t)stream>>>(Fm, okp_epipoles(Fm), left_dev, right_dev, n,
                                                                              round_to_f32, left_out_dev, right_out_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_stereo_associate_f64(const double* F, const double* left_dev, const int32_t* n_left_dev, const double* right_dev,
                             const int32_t* n_right_dev, int B, int max_left, int max_right, double max_distance_px,
                             int32_t* match_dev, double* cost_dev, void* stream) {
    if (B < 0 || max_left < 1 || max_right < 1 || max_left > OKP_ASSOC_MAX || max_right > OKP_ASSOC_MAX) return OKP_E_SHAPE;
    if (B == 0) return OKP_OK;
    if (!F || !left_dev || !n_left_dev || !right_dev || !n_right_dev || !match_dev || !cost_dev) return OKP_E_NULL;
    OkpMat3 Fm;
    for (int i = 0; i < 9; ++i) Fm.m[i] = F[i];
    const size_t smem = sizeof(double) * (size_t)max_left * max_right;
    okp_associate_kernel<<<B, 32, smem, (cudaStream_t)stream>>>(Fm, nullptr, left_dev, n_left_dev, right_dev, n_right_dev,
                                                               max_left, max_right, max_distance_px, match_dev, cost_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_associate_pairs_f64(const double* F_dev, const double* left_dev, const int32_t* n_left_dev, const double* right_dev,
                            const int32_t* n_right_dev, int B, int max_left, int max_right, double max_distance_px,
                            int32_t* match_dev, double* cost_dev, void* stream) {
    if (B < 0 || max_left < 1 || max_right < 1 || max_left > OKP_ASSOC_MAX || max_right > OKP_ASSOC_MAX) return OKP_E_SHAPE;
    if (B == 0) return OKP_OK;
    if (!F_dev || !left_dev || !n_left_dev || !right_dev || !n_right_dev || !match_dev || !cost_dev) return OKP_E_NULL;
    OkpMat3 unused;
    memset(&unused, 0, sizeof(unused));
    const size_t smem = sizeof(double) * (size_t)max_left * max_right;
    okp_associate_kernel<<<B, 32, smem, (cudaStream_t)stream>>>(unused, F_dev, left_dev, n_left_dev, right_dev, n_right_dev,
                                                               max_left, max_right, max_distance_px, match_dev, cost_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

// The object shape the stereo and sequence entries share (params and, for C > 1, keypoint_config checked for NULL):
// O = max_objects and P = 1 + sum(keypoint_config) up to 64, for the greedy step's 64-bit masks.
static int okp_objects_shape(int N, int C, const int32_t* keypoint_config, const OkpDecodeParams* params, OkpStereoShape* shape) {
    OkpStereoShape& d = *shape;
    memset(&d, 0, sizeof(d));
    d.N = N; d.C = C; d.O = params->max_objects;
    if (d.O < 1 || d.O > 64) return OKP_E_SHAPE;                     // the greedy step's 64-bit masks
    d.cfg[0] = 1;
    d.S = 1; d.P = 1;
    for (int c = 1; c < C; ++c) {
        const int k = keypoint_config[c - 1];
        if (k < 1 || k > OKP_MAX_SLOTS) return OKP_E_CAPACITY;
        d.cfg[c] = k; d.off[c] = d.P;
        d.P += k;
        if (k > d.S) d.S = k;
    }
    if (d.P > 64) return OKP_E_SHAPE;
    return OKP_OK;
}

// The host checks and set-up both stereo-objects entries share (after their P = 0 return): NULL pointers, the shape, the rig.
static int okp_stereo_prepare(const OkpDecodeTables* tables, int N, int C, const int32_t* keypoint_config,
                              const OkpDecodeParams* params, const int32_t* pairs_dev, const OkpCamera* left_camera,
                              const OkpCamera* right_camera, const double* F, const double* P_L, const double* P_R,
                              const OkpStereoTables* out, OkpStereoShape* shape, OkpStereoRig* rig_out) {
    if (!tables || !params || (C > 1 && !keypoint_config) || !pairs_dev || !left_camera || !right_camera || !F || !P_L ||
        !P_R || !out)
        return OKP_E_NULL;
    if (!tables->n_objects || !tables->kp_count || !tables->kp_xy || !out->object_match || !out->object_cost ||
        !out->slot_match || !out->point || !out->flags)
        return OKP_E_NULL;
    const int rc = okp_objects_shape(N, C, keypoint_config, params, shape);
    if (rc != OKP_OK) return rc;
    OkpStereoRig& rig = *rig_out;
    rig.cam[0] = *left_camera;
    rig.cam[1] = *right_camera;
    for (int i = 0; i < 9; ++i) rig.F.m[i] = F[i];
    rig.ep = okp_epipoles(rig.F);                                     // as okp_correct_matches_f64 does
    for (int i = 0; i < 12; ++i) { rig.proj[0][i] = P_L[i]; rig.proj[1][i] = P_R[i]; }
    return OKP_OK;
}

int okp_triangulate_stereo_objects_f64(const OkpDecodeTables* tables, int N, int C, const int32_t* keypoint_config,
                                       const OkpDecodeParams* params, const int32_t* pairs_dev, int P,
                                       const OkpCamera* left_camera, const OkpCamera* right_camera, const double* F,
                                       const double* P_L, const double* P_R, double max_distance_px, int optimal_correction,
                                       const OkpStereoTables* out, void* stream) {
    if (N < 0 || P < 0 || C < 1 || C > OKP_MAX_MAPS) return OKP_E_SHAPE;
    if (P == 0) return OKP_OK;
    OkpStereoShape d;
    OkpStereoRig rig;
    const int rc = okp_stereo_prepare(tables, N, C, keypoint_config, params, pairs_dev, left_camera, right_camera, F, P_L, P_R,
                                      out, &d, &rig);
    if (rc != OKP_OK) return rc;
    const size_t smem = okp_stereo_smem_bytes(d.O, d.C, d.P);
    if (smem > 48 * 1024)
        OKP_CUDA_CHECK(cudaFuncSetAttribute(okp_stereo_objects_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    okp_stereo_objects_kernel<<<P, 32, smem, (cudaStream_t)stream>>>(rig, d, tables->n_objects, tables->kp_count, tables->kp_xy,
                                                                     pairs_dev, max_distance_px, optimal_correction, *out);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_triangulate_stereo_objects_depth_f64(const OkpDecodeTables* tables, int N, int C, const int32_t* keypoint_config,
                                             const OkpDecodeParams* params, const int32_t* pairs_dev, int P,
                                             const OkpCamera* left_camera, const OkpCamera* right_camera, const double* F,
                                             const double* P_L, const double* P_R, const double* T_RL,
                                             double max_distance_px, double max_depth_px, int optimal_correction,
                                             const OkpStereoTables* out, void* stream) {
    if (N < 0 || P < 0 || C < 1 || C > OKP_MAX_MAPS) return OKP_E_SHAPE;
    if (P == 0) return OKP_OK;
    OkpStereoShape d;
    OkpStereoRig rig;
    const int rc = okp_stereo_prepare(tables, N, C, keypoint_config, params, pairs_dev, left_camera, right_camera, F, P_L, P_R,
                                      out, &d, &rig);
    if (rc != OKP_OK) return rc;
    if (!T_RL || !tables->kp_point) return OKP_E_NULL;
    if (!(max_depth_px > 0.0 && max_depth_px < INFINITY)) return OKP_E_SHAPE;          // NaN fails both
    const size_t smem = okp_stereo_depth_smem_bytes(d.O, d.C, d.P);
    if (smem > 227 * 1024) return OKP_E_SHAPE;                        // sm_100's per-block opt-in shared memory
    OkpStereoLift lift;
    for (int r = 0; r < 3; ++r) {                                     // [0] = T_RL, [1] = T_LR = T_RL^-1 (a rigid motion)
        for (int c = 0; c < 3; ++c) { lift.R[0][3 * r + c] = T_RL[4 * r + c]; lift.R[1][3 * r + c] = T_RL[4 * c + r]; }
        lift.t[0][r] = T_RL[4 * r + 3];
        lift.t[1][r] = -(T_RL[r] * T_RL[3] + T_RL[4 + r] * T_RL[7] + T_RL[8 + r] * T_RL[11]);
    }
    if (smem > 48 * 1024)
        OKP_CUDA_CHECK(cudaFuncSetAttribute(okp_stereo_depth_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    okp_stereo_depth_kernel<<<P, 32, smem, (cudaStream_t)stream>>>(rig, lift, d, tables->n_objects, tables->kp_count,
                                                                   tables->kp_xy, tables->kp_point, pairs_dev, max_distance_px,
                                                                   max_depth_px, optimal_correction, *out);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_triangulate_sequence_objects_f64(const OkpDecodeTables* tables, int N, int C, const int32_t* keypoint_config,
                                         const OkpDecodeParams* params, const int32_t* frames_dev, int A, int V,
                                         const double* F_dev, const double* motion_dev, const double* poses_dev,
                                         const OkpCamera* camera, int association, double max_distance_px,
                                         double max_depth_px, double max_error_px, int max_rounds,
                                         const OkpSequenceObjectTables* out, void* stream) {
    if (N < 0 || A < 0 || C < 1 || C > OKP_MAX_MAPS) return OKP_E_SHAPE;
    if (A == 0) return OKP_OK;
    if (!tables || !params || (C > 1 && !keypoint_config) || !frames_dev || !F_dev || !poses_dev || !camera || !out)
        return OKP_E_NULL;
    if (!tables->n_objects || !tables->kp_count || !tables->kp_xy || !out->object_match || !out->object_cost ||
        !out->slot_match || !out->flags || !out->observations || !out->valid || !out->observed || !out->point ||
        !out->error || !out->dropped)
        return OKP_E_NULL;
    if (association != 0 && association != 1) return OKP_E_UNSUPPORTED;
    if (association == 1 && (!motion_dev || !tables->kp_point)) return OKP_E_NULL;
    OkpStereoShape d;
    const int rc = okp_objects_shape(N, C, keypoint_config, params, &d);
    if (rc != OKP_OK) return rc;
    // the track kernel's limits (okp_triangulate_tracks_f64), checked here so that nothing is launched before a refusal
    const int Pg = d.O * d.C * d.S;
    if (V < 2 || V > OKP_MAX_VIEWS || max_rounds < 0 || A > 65535 || (long long)A * Pg > 0x7fffffffLL) return OKP_E_SHAPE;
    if (association == 1 && !(max_depth_px > 0.0 && max_depth_px < INFINITY)) return OKP_E_SHAPE;     // NaN fails both
    const size_t smem = okp_sequence_smem_bytes(d.O, d.C, d.P);
    if (smem > 227 * 1024) return OKP_E_SHAPE;                        // sm_100's per-block opt-in shared memory
    if (smem > 48 * 1024)
        OKP_CUDA_CHECK(cudaFuncSetAttribute(okp_sequence_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    okp_sequence_match_kernel<<<A * (V - 1), 32, smem, (cudaStream_t)stream>>>(
        *camera, d, V, tables->n_objects, tables->kp_count, tables->kp_xy, tables->kp_point, frames_dev, F_dev,
        association == 1 ? motion_dev : nullptr, association, max_distance_px, max_depth_px, *out);
    OKP_CUDA_CHECK(cudaGetLastError());
    return okp_triangulate_tracks_f64(out->observations, out->valid, poses_dev, camera, A, Pg, V, max_error_px, max_rounds,
                                      out->point, out->error, out->dropped, stream);
}

int okp_eval_match_f64(const double* kp_point_dev, const int32_t* kp_count_dev, const int32_t* n_objects_dev,
                       const double* T_WC_dev, const double* scene_points_dev, int N, int O, int C, int S, int G, int Kp,
                       const OkpCamera* camera, double frame_limit_x, double frame_limit_y, double max_coordinate,
                       double small_error, int32_t* status_dev, double* gt_point_dev, double* err_dev,
                       double* err_xy_dev, int32_t* gt_object_dev, double* frame_stats_dev, void* stream) {
    if (N < 0 || O < 1 || O > OKP_MAX_OBJECTS || C < 1 || C > OKP_MAX_MAPS || S < 1 || S > OKP_MAX_SLOTS || G < 1 || Kp < 1)
        return OKP_E_SHAPE;
    const size_t smem = sizeof(double) * 3 * (size_t)G * Kp + sizeof(int) * 2 * (size_t)O;
    if (smem > 200 * 1024) return OKP_E_SHAPE;
    if (N == 0) return OKP_OK;
    if (!kp_point_dev || !kp_count_dev || !n_objects_dev || !T_WC_dev || !scene_points_dev || !camera || !status_dev ||
        !gt_point_dev || !err_dev || !err_xy_dev || !gt_object_dev || !frame_stats_dev)
        return OKP_E_NULL;
    OkpEvalDims d;
    d.N = N; d.O = O; d.C = C; d.S = S; d.G = G; d.Kp = Kp;
    auto kernel = okp_eval_match_kernel<128>;
    if (smem > 48 * 1024) OKP_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<N, 128, smem, (cudaStream_t)stream>>>(kp_point_dev, kp_count_dev, n_objects_dev, T_WC_dev, scene_points_dev, d,
                                                    *camera, frame_limit_x, frame_limit_y, max_coordinate, small_error,
                                                    status_dev, gt_point_dev, err_dev, err_xy_dev, gt_object_dev,
                                                    frame_stats_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_eval_summary_f64(const double* frame_stats_dev, int N, double* totals_dev, void* stream) {
    if (N < 0) return OKP_E_SHAPE;
    if (!totals_dev || (N > 0 && !frame_stats_dev)) return OKP_E_NULL;
    okp_eval_summary_kernel<256><<<1, 256, 0, (cudaStream_t)stream>>>(frame_stats_dev, N, totals_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_record_doubles(int O, int C, int S) {
    if (O < 1 || O > OKP_MAX_OBJECTS || C < 1 || C > OKP_MAX_MAPS || S < 1 || S > OKP_MAX_SLOTS) return 0;
    return 2 + O * C + O * C * S * 3;
}

int okp_pack_records_f64(const OkpDecodeTables* tables, int N, int O, int C, int S, long long first_row,
                         double* const* destinations, int n_destinations, void* stream) {
    if (N < 0 || first_row < 0 || okp_record_doubles(O, C, S) == 0) return OKP_E_SHAPE;
    if (n_destinations < 1 || n_destinations > OKP_MAX_PEERS) return OKP_E_SHAPE;
    if (N == 0) return OKP_OK;
    if (!tables || !destinations || !tables->n_objects || !tables->flags || !tables->kp_count || !tables->kp_point)
        return OKP_E_NULL;
    OkpPeerBuffers peers;
    memset(&peers, 0, sizeof(peers));
    for (int d = 0; d < n_destinations; ++d) {
        if (!destinations[d]) return OKP_E_NULL;
        peers.dst[d] = destinations[d];
    }
    const long long total = (long long)N * okp_record_doubles(O, C, S);
    long long blocks = (total + 127) / 128;
    if (blocks > kSmCount * 2) blocks = kSmCount * 2;
    okp_pack_records_kernel<<<(unsigned)blocks, 128, 0, (cudaStream_t)stream>>>(
        tables->n_objects, tables->flags, tables->kp_count, tables->kp_point, N, O * C, O * C * S * 3, first_row,
        n_destinations, peers);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_rasterise_targets_f32(const double* keypoints_dev, const double* depths_dev, const int32_t* n_objects_dev,
                              int N, int G, int C, int H, int W, const int32_t* keypoint_config, int kernel_size,
                              double length_scale, double center_radius, float* heat_dev, float* centers_dev,
                              float* depth_dev, void* stream) {
    int rc = check_shape(N, C, H, W);
    if (rc != OKP_OK) return rc;
    if (G < 1 || G > OKP_MAX_OBJECTS || kernel_size < 0 || !(length_scale > 0.0)) return OKP_E_SHAPE;
    if (N == 0) return OKP_OK;
    if (!keypoints_dev || !depths_dev || !heat_dev || !depth_dev || (C > 1 && (!centers_dev || !keypoint_config)))
        return OKP_E_NULL;
    OkpConfig config;
    memset(&config, 0, sizeof(config));
    config.cfg[0] = 1;                                  // video.py:75: the centre map first
    int Kp = 1;
    for (int i = 0; i < C - 1; ++i) {
        if (keypoint_config[i] < 1 || keypoint_config[i] > OKP_MAX_SLOTS) return OKP_E_CAPACITY;
        config.cfg[1 + i] = keypoint_config[i];
        Kp += keypoint_config[i];
    }
    OkpTargetParams prm;
    prm.kernel_size = kernel_size; prm.length_scale = length_scale; prm.center_radius = center_radius;
    const size_t smem = sizeof(double) * 3 * (size_t)G * Kp;
    auto kernel = okp_rasterise_targets_kernel<256>;
    if (smem > 48 * 1024) OKP_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<(unsigned)((long long)N * C), 256, smem, (cudaStream_t)stream>>>(
        keypoints_dev, depths_dev, n_objects_dev, N, G, Kp, C, H, W, config, prm, heat_dev, centers_dev, depth_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

int okp_scatter_tiles_f32(const float* packed_dev, const int32_t* tile_ids_dev, long long n_tiles, int maps, int H, int W,
                          float* heat_dev, void* stream) {
    if (n_tiles < 0 || maps < 0 || H < 1 || W < 1) return OKP_E_SHAPE;
    if (n_tiles == 0) return OKP_OK;
    if (!packed_dev || !tile_ids_dev || !heat_dev) return OKP_E_NULL;
    if ((uintptr_t)packed_dev & 15u) return OKP_E_UNSUPPORTED;
    const int TX = okp_tiles_x(W), tiles = okp_tiles_y(H) * TX;
    const long long threads = n_tiles * 16;
    okp_scatter_tiles_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        packed_dev, tile_ids_dev, n_tiles, H, W, TX, tiles, heat_dev);
    OKP_CUDA_CHECK(cudaGetLastError());
    return OKP_OK;
}

}  // extern "C"
