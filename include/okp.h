/* okp.h -- C ABI of libokp.so: the B200 (sm_100a) heatmap -> 3D keypoint path.
 *
 * This is the drop-in boundary for the inference hot path of ethz-asl/object_keypoints.
 * The reference has no FFI for this path (it is pure Python on torch-CPU / OpenCV); each
 * entry point below names the reference code it replaces, paths relative to the reference
 * root. INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - plain C types only; every buffer is owned and sized by the caller (PyTorch in this
 *     repo); the library allocates nothing and keeps no global state;
 *   - pointers named *_dev / inside OkpDecodeTables are DEVICE pointers; keypoint_config,
 *     OkpCamera and OkpDecodeParams are read on the HOST at call time; every table array starts
 *     on a 16-byte boundary (OKP_E_UNSUPPORTED otherwise);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*, NULL = default
 *     stream) and the call returns without synchronising;
 *   - return value: OKP_OK or a negative OKP_E_* code (okp_strerror). Data-dependent
 *     conditions (table overflow, outlier votes, ...) are never errors: they are reported per
 *     frame in OkpDecodeTables.flags -- the reference prints them (perception/pipeline.py:123);
 *   - re-entrant: concurrent calls on different streams with different buffers are safe.
 */
#ifndef OKP_H
#define OKP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OKP_VERSION_MAJOR 0
#define OKP_VERSION_MINOR 2

enum {
    OKP_OK = 0,
    OKP_E_NULL = -1,         /* a required pointer is NULL */
    OKP_E_SHAPE = -2,        /* N, C, H, W, P, V ... out of the supported range */
    OKP_E_CAPACITY = -3,     /* max_peaks / max_objects / max_votes out of range */
    OKP_E_UNSUPPORTED = -4,  /* parameter combination not implemented (e.g. nms_size) */
    OKP_E_CUDA = -5,         /* a CUDA runtime call or kernel launch failed */
    OKP_E_WORKSPACE = -6     /* workspace smaller than okp_decode_workspace_bytes() */
};

/* per-frame flag bits in OkpDecodeTables.flags */
#define OKP_FLAG_PEAK_OVERFLOW 1u     /* a map had more peaks than max_peaks; the first max_peaks (raster order) are kept */
#define OKP_FLAG_OBJECT_OVERFLOW 2u   /* more centre peaks than max_objects */
#define OKP_FLAG_OUTLIER_SKIPPED 4u   /* a spoke voted farther than outlier_distance from every centre (pipeline.py:121-124) */
#define OKP_FLAG_CLUSTERED 8u         /* > cfg[t] detections, cfg[t] > 1: merged by k-means (pipeline.py:143-148) */
#define OKP_FLAG_VOTE_OVERFLOW 16u    /* more votes for one object than max_votes */
#define OKP_FLAG_NO_CENTERS 32u       /* empty centre map: frame has no objects (pipeline.py:105-106) */
#define OKP_FLAG_ARGMAX_RESOLVED 64u  /* > cfg[t] detections, cfg[t] == 1: most confident kept (pipeline.py:139-142) */
#define OKP_FLAG_GENERIC_PATH 128u    /* not a property of the data: this call's shape / mode is outside the tuned TMA kernel
                                         (W % 4 != 0, W > 500, 16-bit maps with W % 8 != 0, nms_size 3, box_sum 0) and ran
                                         on the exact generic tile kernels, about 3x slower per pixel -- same results */

#define OKP_MAX_MAPS 16               /* C = 1 + number of keypoint types */
#define OKP_MAX_PEAKS 256             /* upper bound for OkpDecodeParams.max_peaks */
#define OKP_MAX_OBJECTS 128
#define OKP_MAX_SLOTS 8               /* upper bound for any keypoint_config entry */
#define OKP_MAX_VIEWS 64

/* Kalibr pinhole + equidistant camera, as perception/utils/camera_utils.py:7-16,64-81 holds it
 * (K, D, Kinv) plus the clip limits DetectionToPoint.reset derives (pipeline.py:159-162). */
typedef struct OkpCamera {
    double fx, fy, cx, cy;
    double k[4];            /* equidistant distortion k1..k4 */
    double kinv[9];         /* row-major inverse of K, computed by the caller like camera_utils.py:11 */
    int32_t clip_x;         /* int(image_size[0]) - 1: the reference clips x with the HEIGHT (pipeline.py:162,169) */
    int32_t clip_y;         /* int(image_size[1]) - 1 */
} OkpCamera;

typedef struct OkpDecodeParams {
    float threshold;          /* 0.5 on the 5x5 box sum (pipeline.py:73) */
    int32_t nms_size;         /* 5 (perception/models.py:55); 3 = CornerNet's _nms window (py_utils/utils.py:14-19) */
    int32_t box_sum;          /* 1: NMS runs on the 5x5 box sum (pipeline.py:70-72); 0: on the map itself */
    int32_t compat_clip_bug;  /* 1: clip (x, y) with (H-1, W-1) like pipeline.py:169; 0: with (W-1, H-1) */
    double outlier_distance;  /* 20.0 px (pipeline.py:121) */
    int32_t max_peaks;        /* K: peak slots per (frame, map) */
    int32_t max_objects;      /* O: object slots per frame */
    int32_t max_votes;        /* V: vote slots per object */
    int32_t kmeans_iterations;/* Lloyd iterations of the deterministic clustering (default 16) */
    int32_t top_k;            /* 0: every peak, raster order (pipeline.py:73). k > 0: the k highest scores of each map,
                                 score-descending (ties: raster order) -- CornerNet's _topk (py_utils/utils.py:27-38)
                                 per keypoint type; exact when the map has <= max_peaks peaks above the threshold,
                                 otherwise OKP_FLAG_PEAK_OVERFLOW is raised as usual */
    int32_t lean_tables;      /* 0 (default): unused slots of every table are reset (zero / -1) as documented below.
                                 1: only valid slots are written -- peak rows k < min(peak_count, K); kp_assigned / kp_count
                                 rows o < n_objects; kp_peak / kp_xy / kp_point slots s < kp_count; votes v < n_votes --
                                 everything else keeps whatever the buffer held. For callers that read by the counts (the
                                 tables of a 64x64 frame are a quarter of its heatmap bytes: clearing them is the decode's
                                 largest DRAM write). */
    int32_t single_pass;      /* okp_decode_*: 0 (default) = two launches, the peak kernel and then the grouping / 3D lift with
                                 one warp per frame; 1 = ONE streaming pass, the grouping runs in the peak kernel's epilogue
                                 warps straight from the sorted peak list in shared memory (no second kernel re-reads the
                                 peak tables). Same tables either way; the two-launch form is the faster one on a B200
                                 (DESIGN.md section 3), the single pass saves a launch when N is small. */
} OkpDecodeParams;

/* Fixed-capacity structure-of-arrays output. N frames, C maps, K = max_peaks, O = max_objects,
 * S = max(1, max(keypoint_config)), V = max_votes. Map 0 is the object-centre map. All arrays are
 * dense row-major with the shapes given; unused slots are zero / -1 (unless OkpDecodeParams.lean_tables). */
typedef struct OkpDecodeTables {
    /* peaks of every map, raster (row-major y, x) order -- pipeline.py:69-79 */
    int32_t* peak_count;    /* [N,C]      true number of peaks (may exceed K) */
    int32_t* peak_yx;       /* [N,C,K,2]  pixel (y, x) */
    float*   peak_score;    /* [N,C,K]    5x5 box sum at the peak */
    float*   peak_xy;       /* [N,C,K,2]  centroid (x, y), pixel-index coordinates (pipeline.py:59,76) */
    float*   peak_conf;     /* [N,C,K]    sum of the window's probabilities (pipeline.py:61) */
    /* spoke -> object assignment -- pipeline.py:115-128 */
    int32_t* peak_object;   /* [N,C,K]    object index, -1 = skipped or no centres */
    double*  peak_vote;     /* [N,C,K,2]  predicted centre (x, y) */
    /* objects -- pipeline.py:130-152,189-199 */
    int32_t* n_objects;     /* [N] */
    uint32_t* flags;        /* [N]        OKP_FLAG_* */
    int32_t* kp_assigned;   /* [N,O,C]    detections assigned before resolution */
    int32_t* kp_count;      /* [N,O,C]    keypoints kept: 1 for the centre, <= keypoint_config[c-1] otherwise */
    int32_t* kp_peak;       /* [N,O,C,S]  index into the map's peak list, -1 for cluster centres */
    float*   kp_xy;         /* [N,O,C,S,2] */
    double*  kp_point;      /* [N,O,C,S,3] camera-frame point 'p_C' (pipeline.py:164-171) */
    int32_t* n_votes;       /* [N,O] */
    double*  votes;         /* [N,O,V,2]  'p_centers' in assignment order */
} OkpDecodeTables;

int okp_version(void);
const char* okp_strerror(int code);

/* Scratch bytes okp_decode_* / okp_extract_peaks_* need for this problem size (either element type): the tile lists of the
 * overflow fix-up and the counter the peak kernel's CTAs claim their work from. The contents need no initialisation and
 * mean nothing between calls, but two calls that may run concurrently (different streams) need different workspaces. */
size_t okp_decode_workspace_bytes(int N, int C, int H, int W, const OkpDecodeParams* params);

/* Replaces KeypointExtractionComponent.__call__ (perception/pipeline.py:64-91) including
 * perception/models.py:55-58 (nms): box sum, NMS, threshold, raster-order compaction and
 * sub-pixel centroid for every map of every frame. Fills the peak_* tables (peak_object and
 * peak_vote are reset). heat_dev: [N,C,H,W] float32 probabilities.
 * The reference's configuration (nms_size 5, box_sum 1, top_k 0) runs on the tuned TMA kernel; the other
 * combinations (3x3 window, NMS on the raw map, per-type top-k: BASELINE.json's "3x3 max-pool NMS ... with
 * per-type top-k and thresholding") run on the exact generic tile kernels. */
int okp_extract_peaks_f32(const float* heat_dev, int N, int C, int H, int W,
                          const OkpDecodeParams* params, const OkpDecodeTables* tables,
                          void* workspace_dev, size_t workspace_bytes, void* stream);

/* okp_extract_peaks_f32 with two optional CUDA events (cudaEvent_t passed as void*, NULL = none) recorded on `stream` right
 * before and right after the peak kernel itself -- i.e. without the work counter's memset in front of it and the overflow
 * fix-up behind it: for callers that time the kernel (bench.py's roofline figure). Same work, same tables. */
int okp_extract_peaks_events_f32(const float* heat_dev, int N, int C, int H, int W,
                                 const OkpDecodeParams* params, const OkpDecodeTables* tables,
                                 void* workspace_dev, size_t workspace_bytes, void* event_before, void* event_after,
                                 void* stream);

/* Replaces ObjectExtraction.__call__ (pipeline.py:104-153) and the DetectionToPoint loop of
 * ObjectKeypointPipeline.__call__ (pipeline.py:189-199, 164-171; camera_utils.py:31-34,75-81)
 * for every frame, reading the peak_* tables. depth_dev [N,C,H,W], centers_dev [N,C-1,2,H,W]:
 * device memory or okp_host_alias() of pinned host memory (gather-only, see below).
 * camera may be NULL: then kp_point is left zero (ObjectExtraction only). */
int okp_group_objects_f32(const float* depth_dev, const float* centers_dev, int N, int C, int H, int W,
                          const int32_t* keypoint_config, const OkpCamera* camera,
                          const OkpDecodeParams* params, const OkpDecodeTables* tables, void* stream);

/* Device-side alias of a page-locked HOST buffer (cudaHostAlloc / cudaHostRegister, e.g. a
 * torch pinned tensor). okp_group_objects_f32 only GATHERS from depth and centers (3 floats per
 * spoke peak), so a caller holding those maps in pinned host memory -- the reference hands
 * ObjectKeypointPipeline.__call__ CPU tensors, pipeline.py:24-28,184-186 -- passes the alias as
 * depth_dev / centers_dev instead of copying 2/3 of the frame's bytes to HBM. Writes the alias to
 * *dev_ptr_out; OKP_E_UNSUPPORTED if the buffer is pageable or not mapped into the current device. */
int okp_host_alias(const void* host_ptr, void** dev_ptr_out);

/* Replaces ObjectKeypointPipeline.__call__ (pipeline.py:182-200) for a batch of N frames:
 * okp_extract_peaks_f32 followed by okp_group_objects_f32 on the same stream (two launches plus the overflow fix-up,
 * which is a no-op unless a map overflowed max_peaks). With OkpDecodeParams.single_pass, for the reference's
 * configuration (nms_size 5, box_sum 1, top_k 0) on shapes the TMA kernel covers, ONE streaming pass instead: the
 * grouping and the 3D lift of a frame run in the epilogue warps of the peak kernel, from the frame's peak list in
 * shared memory, while the next frames stream. Same tables either way. heat_dev must be 16-byte aligned
 * (OKP_E_UNSUPPORTED otherwise). */
int okp_decode_f32(const float* heat_dev, const float* depth_dev, const float* centers_dev,
                   int N, int C, int H, int W, const int32_t* keypoint_config,
                   const OkpCamera* camera, const OkpDecodeParams* params,
                   const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes,
                   void* stream);

/* bfloat16 forms of the three decode entries, for network heads that write bf16 (BASELINE config 5:
 * the reference's InferenceComponent, pipeline.py:13-28, hands over whatever dtype the TorchScript
 * model produces; package_model.py:28 applies the sigmoid inside the model). All three maps are bf16
 * [same shapes as the _f32 forms]; bf16 -> float32 is exact and every sum, comparison and centroid is
 * computed in float32 exactly as in the _f32 forms, so the tables equal those of the _f32 entry run on
 * the up-cast maps bit for bit. The TMA path needs W % 8 == 0; other widths take the generic kernels. */
int okp_extract_peaks_bf16(const void* heat_dev, int N, int C, int H, int W,
                           const OkpDecodeParams* params, const OkpDecodeTables* tables,
                           void* workspace_dev, size_t workspace_bytes, void* stream);
int okp_group_objects_bf16(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                           const int32_t* keypoint_config, const OkpCamera* camera,
                           const OkpDecodeParams* params, const OkpDecodeTables* tables, void* stream);
int okp_decode_bf16(const void* heat_dev, const void* depth_dev, const void* centers_dev,
                    int N, int C, int H, int W, const int32_t* keypoint_config,
                    const OkpCamera* camera, const OkpDecodeParams* params,
                    const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes,
                    void* stream);

/* float16 forms of the same entries, for heads that write float16 (torch.autocast on CUDA, model.half(), a half-precision
 * TorchScript export). All three maps are float16 [same shapes as the _f32 forms]; every float16 value, subnormals
 * included, is exactly a float32 value, and every sum, comparison and centroid is computed in float32 exactly as in the
 * _f32 forms, so the tables equal those of the _f32 entry run on the up-cast maps bit for bit. The TMA path needs
 * W % 8 == 0; other widths take the generic kernels. */
int okp_extract_peaks_f16(const void* heat_dev, int N, int C, int H, int W,
                          const OkpDecodeParams* params, const OkpDecodeTables* tables,
                          void* workspace_dev, size_t workspace_bytes, void* stream);
int okp_group_objects_f16(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                          const int32_t* keypoint_config, const OkpCamera* camera,
                          const OkpDecodeParams* params, const OkpDecodeTables* tables, void* stream);
int okp_decode_f16(const void* heat_dev, const void* depth_dev, const void* centers_dev,
                   int N, int C, int H, int W, const int32_t* keypoint_config,
                   const OkpCamera* camera, const OkpDecodeParams* params,
                   const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes,
                   void* stream);

/* okp_decode_* that also EMITS one compact record per frame -- what ObjectKeypointPipeline.__call__ returns per
 * frame (pipeline.py:195-199): object count, kept-keypoint counts, camera-frame 3D points -- into every sink buffer
 * while it decodes. This is the multi-GPU exchange of SURVEY section 8e (the reference is single-GPU, batch 1:
 * pipeline.py:183): frames shard independently, the only cross-GPU step is the gather of these records. With the
 * peer-mapped (symmetric-memory) buffer of the gathering rank as sink the stores travel over NVLink / NVSwitch from
 * inside the decode kernel -- there is no exchange kernel; the caller provides the cross-rank barrier before the
 * buffer is read. Record layout (little endian, `record_bytes` apart, row first_row + n for frame n):
 *     int32 n_objects; uint32 flags; int32 kp_count[O][C]; (pad to 8); double point[O][P][3]
 * with O = max_objects, P = 1 + sum(keypoint_config): object o's points in (map, slot) order. Only rows o < n_objects
 * and slots s < kp_count[o][c] are written. okp_record_bytes() is the minimum record_bytes. */
typedef struct OkpRecordSink {
    void* const* buffers_dev;   /* HOST array of n_buffers <= 16 DEVICE pointers to [rows, record_bytes] byte buffers */
    int32_t n_buffers;          /* 0: no records (the call is okp_decode_*) */
    int32_t record_bytes;
    long long first_row;
} OkpRecordSink;
int okp_record_bytes(int O, int C, const int32_t* keypoint_config);
int okp_decode_emit_f32(const float* heat_dev, const float* depth_dev, const float* centers_dev,
                        int N, int C, int H, int W, const int32_t* keypoint_config,
                        const OkpCamera* camera, const OkpDecodeParams* params,
                        const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes,
                        const OkpRecordSink* sink, void* stream);
int okp_decode_emit_bf16(const void* heat_dev, const void* depth_dev, const void* centers_dev,
                         int N, int C, int H, int W, const int32_t* keypoint_config,
                         const OkpCamera* camera, const OkpDecodeParams* params,
                         const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes,
                         const OkpRecordSink* sink, void* stream);
int okp_decode_emit_f16(const void* heat_dev, const void* depth_dev, const void* centers_dev,
                        int N, int C, int H, int W, const int32_t* keypoint_config,
                        const OkpCamera* camera, const OkpDecodeParams* params,
                        const OkpDecodeTables* tables, void* workspace_dev, size_t workspace_bytes,
                        const OkpRecordSink* sink, void* stream);
/* okp_group_objects_* with the record sink of okp_decode_emit_*: the second half of the two-launch decode for callers
 * that run the halves themselves (e.g. to put an event between them; ObjectExtraction + DetectionToPoint,
 * pipeline.py:104-171,189-199). sink may be NULL. */
int okp_group_objects_emit_f32(const float* depth_dev, const float* centers_dev, int N, int C, int H, int W,
                               const int32_t* keypoint_config, const OkpCamera* camera,
                               const OkpDecodeParams* params, const OkpDecodeTables* tables,
                               const OkpRecordSink* sink, void* stream);
int okp_group_objects_emit_bf16(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                                const int32_t* keypoint_config, const OkpCamera* camera,
                                const OkpDecodeParams* params, const OkpDecodeTables* tables,
                                const OkpRecordSink* sink, void* stream);
int okp_group_objects_emit_f16(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                               const int32_t* keypoint_config, const OkpCamera* camera,
                               const OkpDecodeParams* params, const OkpDecodeTables* tables,
                               const OkpRecordSink* sink, void* stream);

/* Per-frame cameras: okp_decode_emit_* / okp_group_objects_emit_* for a batch whose frames come from more than one camera
 * (the two views of a stereo rig, sequences with different calibrations or different crops). Frame n is undistorted,
 * clipped (clip_x / clip_y) and unprojected with cameras_dev[n]; everything else is the single-camera entry's
 * arithmetic, so the rows of frame n equal that entry's rows for the same frame run with camera = &cameras_dev[n].
 * cameras_dev: DEVICE array [N] of OkpCamera (144 bytes each), 16-byte aligned, read by the grouping kernel (one load
 * per frame). It is a device pointer because a caller reuses one table for every batch of the same layout; the indices
 * behind it are the caller's to check. sink may be NULL. N = 0 returns OKP_OK, as for every entry. With N > 0, refused on
 * the host, before any CUDA call: NULL cameras_dev or NULL depth_dev (OKP_E_NULL), cameras_dev not 16-byte aligned or
 * OkpDecodeParams.single_pass set (OKP_E_UNSUPPORTED: only the two-launch form has a per-frame camera). */
int okp_decode_cameras_f32(const float* heat_dev, const float* depth_dev, const float* centers_dev,
                           int N, int C, int H, int W, const int32_t* keypoint_config,
                           const OkpCamera* cameras_dev /* DEVICE [N]: frame n is lifted with cameras_dev[n] */,
                           const OkpDecodeParams* params, const OkpDecodeTables* tables, void* workspace_dev,
                           size_t workspace_bytes, const OkpRecordSink* sink, void* stream);
int okp_decode_cameras_bf16(const void* heat_dev, const void* depth_dev, const void* centers_dev,
                            int N, int C, int H, int W, const int32_t* keypoint_config, const OkpCamera* cameras_dev,
                            const OkpDecodeParams* params, const OkpDecodeTables* tables, void* workspace_dev,
                            size_t workspace_bytes, const OkpRecordSink* sink, void* stream);
int okp_decode_cameras_f16(const void* heat_dev, const void* depth_dev, const void* centers_dev,
                           int N, int C, int H, int W, const int32_t* keypoint_config, const OkpCamera* cameras_dev,
                           const OkpDecodeParams* params, const OkpDecodeTables* tables, void* workspace_dev,
                           size_t workspace_bytes, const OkpRecordSink* sink, void* stream);
int okp_group_objects_cameras_f32(const float* depth_dev, const float* centers_dev, int N, int C, int H, int W,
                                  const int32_t* keypoint_config, const OkpCamera* cameras_dev,
                                  const OkpDecodeParams* params, const OkpDecodeTables* tables,
                                  const OkpRecordSink* sink, void* stream);
int okp_group_objects_cameras_bf16(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                                   const int32_t* keypoint_config, const OkpCamera* cameras_dev,
                                   const OkpDecodeParams* params, const OkpDecodeTables* tables,
                                   const OkpRecordSink* sink, void* stream);
int okp_group_objects_cameras_f16(const void* depth_dev, const void* centers_dev, int N, int C, int H, int W,
                                  const int32_t* keypoint_config, const OkpCamera* cameras_dev,
                                  const OkpDecodeParams* params, const OkpDecodeTables* tables,
                                  const OkpRecordSink* sink, void* stream);

/* Replaces FisheyeCamera.undistort (camera_utils.py:75-81, cv2.fisheye.undistortPoints with
 * P = K). xy_dev/out_dev: [n,2] float64. round_to_f32 != 0 reproduces OpenCV's float32 output
 * for float32 input (the value is rounded to float32, stored as float64). */
int okp_fisheye_undistort_f64(const double* xy_dev, int n, const OkpCamera* camera,
                              int round_to_f32, double* out_dev, void* stream);

/* Replaces FisheyeCamera.project (camera_utils.py:65-73, cv2.fisheye.projectPoints).
 * X_dev [n,3] float64 world points, T_CW: 16 doubles row-major on the HOST, out_dev [n,2]. */
int okp_fisheye_project_f64(const double* X_dev, int n, const double* T_CW, const OkpCamera* camera,
                            double* out_dev, void* stream);

/* Replaces DetectionToPoint.__call__ (pipeline.py:164-171): undistort, round, clip, depth lookup,
 * unproject. xy_dev [n,2] float32, depth_map_dev [H,W] float32, out_dev [n,3] float64. */
int okp_detection_to_point_f32(const float* xy_dev, int n, const float* depth_map_dev, int H, int W,
                               const OkpCamera* camera, const OkpDecodeParams* params,
                               double* out_dev, void* stream);

/* Batched multi-view DLT. Replaces the cv2.triangulatePoints calls of StereoCamera.triangulate
 * (camera_utils.py:103-108) and LabelingApp._triangulate (scripts/label.py:296-305) and
 * generalises them to V views. points_dev [P,V,2] float64 UNDISTORTED pixels, valid_dev [P,V]
 * uint8 (NULL = all valid), projections_dev [V,3,4] float64 when per_point_projections == 0,
 * else [P,V,3,4]. out_dev [P,3]; points with fewer than two valid views get NaN. */
int okp_triangulate_f64(const double* points_dev, const uint8_t* valid_dev,
                        const double* projections_dev, int per_point_projections, int P, int V,
                        double* out_dev, void* stream);

/* Reprojection-error filter (absent from the reference as code; north_star names it): project
 * X_dev [P,3] into every view (poses_dev [V,4,4] world->camera float64, one equidistant camera),
 * write the pixel error err_dev [P,V] against the DISTORTED observations obs_dev [P,V,2], and clear
 * valid_dev[p,v] where the error exceeds max_error_px. */
int okp_reprojection_filter_f64(const double* X_dev, const double* obs_dev, uint8_t* valid_dev,
                                const double* poses_dev, const OkpCamera* camera, int P, int V,
                                double max_error_px, double* err_dev, void* stream);

/* Robust multi-view triangulation, K5 and K6 fused (north_star: "batched multi-view DLT ... and
 * reprojection-error filtering"; the reference stops at two views, scripts/label.py:285-305).
 * Per point: undistort the valid observations (camera_utils.py:75-81), V-view DLT with the
 * projections K * poses[v][:3] (camera_utils.py:125-130), reprojection error of every view; while
 * the worst valid view is farther than max_error_px, more than two views remain and fewer than
 * max_rounds views were dropped: drop it and solve again. obs_dev [P,V,2] DISTORTED pixels,
 * valid_dev [P,V] in/out (NULL = all valid, nothing written back), poses_dev [V,4,4] world->camera,
 * out_dev [P,3], err_dev [P,V] error against the final point, dropped_dev [P] (may be NULL). */
int okp_triangulate_robust_f64(const double* obs_dev, uint8_t* valid_dev, const double* poses_dev,
                               const OkpCamera* camera, int P, int V, double max_error_px, int max_rounds,
                               double* out_dev, double* err_dev, int32_t* dropped_dev, void* stream);

/* okp_triangulate_robust_f64 for TRACKS of a moving camera (BASELINE config 3: a 30 s sequence, 16 viewpoints per point):
 * the points come in G groups of Pg, each group seen from its own V poses -- the generalisation of
 * LabelingApp._triangulate (scripts/label.py:285-305: one pose pair per labelled point) to V views. obs_dev [G,Pg,V,2],
 * valid_dev [G,Pg,V], poses_dev [G,V,4,4] world->camera, out_dev [G,Pg,3], err_dev [G,Pg,V], dropped_dev [G,Pg]. */
int okp_triangulate_tracks_f64(const double* obs_dev, uint8_t* valid_dev, const double* poses_dev,
                               const OkpCamera* camera, int G, int Pg, int V, double max_error_px, int max_rounds,
                               double* out_dev, double* err_dev, int32_t* dropped_dev, void* stream);

/* Replaces the cv2.correctMatches call of StereoCamera.triangulate (camera_utils.py:100-101): the
 * Hartley-Sturm optimal correction. F: 9 doubles row-major on the HOST with x_right^T F x_left = 0
 * (camera_utils.py:184-189). left_dev/right_dev: [n,2] float64 UNDISTORTED pixels; the outputs are the
 * closest pair (in summed squared pixel distance) that satisfies the epipolar constraint exactly.
 * round_to_f32 != 0 rounds the outputs to float32 like OpenCV does for the float32 input the
 * reference passes (camera_utils.py:93-94). Where the minimum is at t = infinity OpenCV returns NaN;
 * this entry returns the limit point. */
int okp_correct_matches_f64(const double* F, const double* left_dev, const double* right_dev, int n,
                            int round_to_f32, double* left_out_dev, double* right_out_dev, void* stream);

/* Stereo association (the AssociationComponent test/test_pipeline.py:208-261 expects; its
 * implementation is absent from the reference). For each of B frame pairs: left_dev [B,max_left,2] and
 * right_dev [B,max_right,2] float64 UNDISTORTED pixels with n_left_dev / n_right_dev [B] valid counts
 * (max_left, max_right <= 64). cost = mean of the two point-to-epipolar-line distances; matches are
 * taken greedily by globally smallest cost, one-to-one, while cost <= max_distance_px.
 * match_dev [B,max_left]: index into the frame's right points or -1; cost_dev [B,max_left]. */
int okp_stereo_associate_f64(const double* F, const double* left_dev, const int32_t* n_left_dev,
                             const double* right_dev, const int32_t* n_right_dev, int B, int max_left,
                             int max_right, double max_distance_px, int32_t* match_dev, double* cost_dev,
                             void* stream);

/* okp_stereo_associate_f64 with one fundamental matrix PER PAIR, F_dev [B,9] in device memory: association between two
 * frames of a moving camera, whose F follows from the two poses (scripts/label.py:285-297 builds exactly that pair
 * geometry for its two-view triangulation). */
int okp_associate_pairs_f64(const double* F_dev, const double* left_dev, const int32_t* n_left_dev,
                            const double* right_dev, const int32_t* n_right_dev, int B, int max_left,
                            int max_right, double max_distance_px, int32_t* match_dev, double* cost_dev,
                            void* stream);

/* Stereo objects: the decoded objects of P frame pairs of one stereo rig, matched across the two views and triangulated in
 * the left camera's frame. O = max_objects, S = max(1, max(keypoint_config)) as in OkpDecodeTables; all arrays are device
 * memory, dense row-major with the shapes given, and every entry is written. */
#define OKP_STEREO_AMBIGUOUS 1u   /* a left object had two or more right objects within max_distance_px before the greedy
                                     step: objects on one epipolar line, which epipolar matching cannot tell apart */
#define OKP_STEREO_BAD_PAIR 2u    /* a frame index of the pair is outside [0, N): nothing was read or matched */
#define OKP_STEREO_NO_DEPTH 4u    /* depth association only: a candidate within max_distance_px had no valid lift in
                                     either view, and was not matched */
typedef struct OkpStereoTables {
    int32_t* object_match;  /* [P,O]       right object of left object o, -1 */
    double*  object_cost;   /* [P,O]       epipolar cost of that match (pixels), 0 where there is none */
    int32_t* slot_match;    /* [P,O,C,S]   right object's slot matched to left slot s, -1 */
    double*  point;         /* [P,O,C,S,3] left camera frame, NaN where slot_match is -1 */
    uint32_t* flags;        /* [P]         OKP_STEREO_* */
} OkpStereoTables;

/* For each pair p = (l, r) = (pairs_dev[2p], pairs_dev[2p+1]) of frames of `tables` (N frames decoded with C maps,
 * keypoint_config and params; lean tables or cleared ones, only valid slots are read):
 *   1. every valid keypoint kp_xy[f,o,c,s] (s < kp_count) of both frames is undistorted with its view's camera;
 *   2. objects are matched by their centre keypoints with the cost and greedy one-to-one rule of okp_stereo_associate_f64
 *      (mean point-to-epipolar-line distance, globally smallest first, ties to the smaller left then right index, while
 *      cost <= max_distance_px);
 *   3. for each matched object pair and each spoke type c >= 1 the two objects' slots of type c are matched the same way
 *      (the centre slot is matched with its object);
 *   4. every matched keypoint pair is triangulated like StereoCamera.triangulate (camera_utils.py:92-110): undistorted
 *      points rounded to float32, with optimal_correction the Hartley-Sturm correction of okp_correct_matches_f64 rounded
 *      to float32, then the two-view DLT with P_L, P_R, dehomogenised.
 * F, P_L, P_R: 9, 12, 12 doubles row-major on the HOST (StereoCamera.F with x_R^T F x_L = 0, and
 * StereoCamera.projection_matrices: K_L [I|0], K_R T_RL[:3]). pairs_dev: DEVICE int32 [P,2]; a pair with an index
 * outside [0, N) gets OKP_STEREO_BAD_PAIR. P = 0 returns OKP_OK. Refused on the host, before any CUDA call: NULL pointers
 * (OKP_E_NULL); N < 0, P < 0, C out of range, max_objects > 64 or 1 + sum(keypoint_config) > 64 (OKP_E_SHAPE: the greedy
 * step keeps its used rows and columns in 64-bit masks). */
int okp_triangulate_stereo_objects_f64(const OkpDecodeTables* tables, int N, int C, const int32_t* keypoint_config,
                                       const OkpDecodeParams* params, const int32_t* pairs_dev, int P,
                                       const OkpCamera* left_camera, const OkpCamera* right_camera, const double* F,
                                       const double* P_L, const double* P_R, double max_distance_px, int optimal_correction,
                                       const OkpStereoTables* out, void* stream);

/* okp_triangulate_stereo_objects_f64 with depth association: objects on one epipolar line (side by side in the same
 * image rows of this kind of rig) are told apart by each view's monocular lift, tables->kp_point (the frame's own camera
 * frame: decode with a camera table). Per pair, the lift X of every valid keypoint is projected into the other view,
 * q_R = pi(K_R (R_RL X_L + t_RL)) and q_L = pi(K_L (R_LR X_R + t_LR)) with T_LR = T_RL^-1 and K from fx, fy, cx, cy of
 * the camera; a lift is valid when it is finite with z > 0. A candidate (i, j) is admissible when its epipolar cost (as
 * above) is <= max_distance_px and d(i, j) <= max_depth_px, d = 0.5 (|q_R(i) - u_R(j)| + |q_L(j) - u_L(i)|) over the
 * undistorted pixels u, or the one term whose lift is valid. The greedy one-to-one step of steps 2 and 3 runs on d over
 * the admissible candidates (same tie rule); steps 1 and 4 are unchanged, and object_cost holds d. A candidate within
 * max_distance_px without a valid lift on either side is never matched and sets OKP_STEREO_NO_DEPTH; OKP_STEREO_AMBIGUOUS
 * marks a pair in which a left object had two or more admissible right objects.
 * T_RL: 16 doubles row-major on the HOST (StereoCamera.T_RL, left camera frame -> right camera frame).
 * P = 0 returns OKP_OK. Refused on the host, before any CUDA call: every refusal of okp_triangulate_stereo_objects_f64;
 * NULL T_RL or NULL tables->kp_point (OKP_E_NULL); max_depth_px not finite or <= 0 (OKP_E_SHAPE); a shape whose shared
 * memory, 8 (8 O P + O^2 + 64) + 5 O P + O + 2 O C bytes, exceeds sm_100's 227 KB per-block limit (OKP_E_SHAPE). */
int okp_triangulate_stereo_objects_depth_f64(const OkpDecodeTables* tables, int N, int C, const int32_t* keypoint_config,
                                             const OkpDecodeParams* params, const int32_t* pairs_dev, int P,
                                             const OkpCamera* left_camera, const OkpCamera* right_camera, const double* F,
                                             const double* P_L, const double* P_R, const double* T_RL,
                                             double max_distance_px, double max_depth_px, int optimal_correction,
                                             const OkpStereoTables* out, void* stream);

/* Sequence objects: the decoded objects of a sequence filmed by one moving camera with known poses (BASELINE config 3),
 * each anchor frame's objects matched into its V - 1 view frames and every anchor keypoint triangulated over the views
 * in the world frame. A anchors, O = max_objects, S = max(1, max(keypoint_config)); all arrays are device memory, dense
 * row-major with the shapes given, and every entry is written. */
typedef struct OkpSequenceObjectTables {
    int32_t* object_match;  /* [A,V-1,O]       object of view frame v + 1 matched to anchor object o, -1 */
    double*  object_cost;   /* [A,V-1,O]       cost of that match (epipolar cost, or d with depth association), 0 where none */
    int32_t* slot_match;    /* [A,V-1,O,C,S]   matched object's slot for anchor slot s, -1 */
    uint32_t* flags;        /* [A,V-1]         OKP_STEREO_* of the pair (anchor, view v + 1) */
    double*  observations;  /* [A,O,C,S,V,2]   track of every anchor slot: view 0 the anchor's keypoint, view v its match in
                               view frame v; kp_xy (distorted pixels), 0 where there is none */
    uint8_t* valid;         /* [A,O,C,S,V]     observed, after the reprojection filter */
    uint8_t* observed;      /* [A,O,C,S,V]     1 where the track has an observation */
    double*  point;         /* [A,O,C,S,3]     world frame, NaN where fewer than two views are valid */
    double*  error;         /* [A,O,C,S,V]     reprojection error (pixels) against the final point; NaN for a track with
                               fewer than two observations */
    int32_t* dropped;       /* [A,O,C,S]       views dropped by the reprojection filter */
} OkpSequenceObjectTables;

/* For every anchor a and view v in [1, V): the pair (anchor frame frames_dev[a,0], view frame frames_dev[a,v]) of `tables`
 * (N frames decoded with C maps, keypoint_config and params, all with `camera`; lean tables or cleared ones, only valid
 * slots are read) is matched like a stereo pair of okp_triangulate_stereo_objects_f64 (association 0: epipolar cost under
 * F_dev[a,v-1], <= max_distance_px) or of okp_triangulate_stereo_objects_depth_f64 (association 1: kp_point lifts projected
 * with the pair's rigid motion, epipolar gate, then d <= max_depth_px), anchor frame as the left view: objects by their
 * centres, then each matched object pair's slots type by type; same costs, tie rule and flags. Every anchor slot's matches
 * form a track of V views, which okp_triangulate_tracks_f64 solves with G = A groups of O*C*S tracks: undistortion, V-view
 * DLT with the poses poses_dev[a], reprojection filter with max_error_px and max_rounds, world-frame points.
 * frames_dev: DEVICE int32 [A,V]. F_dev: DEVICE [A,V-1,3,3] row-major, x_view^T F x_anchor = 0 for undistorted pixels.
 * motion_dev: DEVICE [A,V-1,2,12]: (R row-major, t) of T = T_CW[view] T_CW[anchor]^-1 (anchor camera -> view camera), then
 * (R^T, -R^T t); read with association 1 only (may be NULL otherwise). poses_dev: DEVICE [A,V,4,4] world -> camera of the
 * frames. A pair with a frame index outside [0, N) gets OKP_STEREO_BAD_PAIR and matches nothing (column 0 still holds the
 * anchor's keypoints when the anchor frame is in range). A = 0 returns OKP_OK. Refused on the host, before any CUDA call:
 * NULL pointers (OKP_E_NULL; with association 1 also NULL motion_dev or tables->kp_point); association not 0 or 1
 * (OKP_E_UNSUPPORTED); N < 0, A < 0, C out of range, max_objects > 64, 1 + sum(keypoint_config) > 64, V < 2, V > 64,
 * A > 65535, A * O * C * S > 2^31 - 1, max_rounds < 0, a max_depth_px (association 1) not finite or <= 0, or a shape whose
 * shared memory, 8 (8 O P + O^2 + 64) + O P + O + 2 O C bytes with P = 1 + sum(keypoint_config), exceeds sm_100's 227 KB
 * per-block limit (OKP_E_SHAPE). */
int okp_triangulate_sequence_objects_f64(const OkpDecodeTables* tables, int N, int C, const int32_t* keypoint_config,
                                         const OkpDecodeParams* params, const int32_t* frames_dev, int A, int V,
                                         const double* F_dev, const double* motion_dev, const double* poses_dev,
                                         const OkpCamera* camera, int association, double max_distance_px,
                                         double max_depth_px, double max_error_px, int max_rounds,
                                         const OkpSequenceObjectTables* out, void* stream);

/* Evaluation bookkeeping (SURVEY section 8f rank 3). Replaces Results.add of the reference's
 * scripts/eval_model.py:141-187 for a batch of N frames, reading the decode tables in place:
 * kp_point_dev [N,O,C,S,3], kp_count_dev [N,O,C], n_objects_dev [N] (OkpDecodeTables fields), T_WC_dev
 * [N,4,4] camera->world per frame, scene_points_dev [G,Kp,3] world points, row 0 of each object its centre
 * (perception/datasets/video.py:121-129). Every predicted object is matched to the ground-truth object with
 * the nearest centre in camera-frame XY (:153-155) and dropped when that centre does not project into the
 * frame (:158-163); a point with all coordinates < max_coordinate (2.0) is matched to the nearest of the
 * object's ground-truth points (:171-173) and dropped when that point is not in view (:174-178), any other
 * point counts as missing (:183-185). frame_limit_x / frame_limit_y are camera.image_size[0] / [1] AS THE
 * REFERENCE HOLDS THEM, i.e. (H, W) compared with (x, y) (camera_utils.py:36-43).
 * Outputs: status_dev [N,O,C,S] (-1 empty slot, 0 matched, 1 missing, 2 point not in view, 3 object not in
 * view), gt_point_dev [N,O,C,S,3] camera-frame ground truth, err_dev / err_xy_dev [N,O,C,S] metres,
 * gt_object_dev [N,O], frame_stats_dev [N,8] per-frame (matched, missing, errors < small_error, mean, M2,
 * sum of xy errors, 0, 0) for okp_eval_summary_f64. */
int okp_eval_match_f64(const double* kp_point_dev, const int32_t* kp_count_dev, const int32_t* n_objects_dev,
                       const double* T_WC_dev, const double* scene_points_dev, int N, int O, int C, int S,
                       int G, int Kp, const OkpCamera* camera, double frame_limit_x, double frame_limit_y,
                       double max_coordinate, double small_error, int32_t* status_dev, double* gt_point_dev,
                       double* err_dev, double* err_xy_dev, int32_t* gt_object_dev, double* frame_stats_dev,
                       void* stream);

/* Replaces the accumulation loop of Results.print_results (scripts/eval_model.py:192-214): merges
 * frame_stats_dev [N,8] into totals_dev [8] = (matched, missing, small, mean error, M2 = sum of squared
 * deviations, sum of xy errors, 0, 0), metres, deterministically (fixed merge order). */
int okp_eval_summary_f64(const double* frame_stats_dev, int N, double* totals_dev, void* stream);

/* Multi-GPU exchange (SURVEY section 8e; the reference is single-GPU, batch 1: pipeline.py:183). Frames
 * shard independently; the only cross-GPU step is the gather of the per-frame 3D keypoint records. A record
 * is okp_record_doubles(O, C, S) = 2 + O*C + O*C*S*3 float64: n_objects, flags, kp_count[O,C],
 * kp_point[O,C,S,3] -- what ObjectKeypointPipeline.__call__ returns per frame (pipeline.py:195-199). */
int okp_record_doubles(int O, int C, int S);

/* Packs the N records of `tables` and stores them at rows [first_row, first_row + N) of every destination
 * buffer (`destinations`: HOST array of n_destinations <= 16 DEVICE pointers to [rows, R] float64 buffers).
 * One destination = the pack step in front of an NCCL all_gather. With the peer-mapped buffers of all ranks
 * as destinations (first_row = rank * N) this call is the all_gather itself: the stores go over NVLink
 * while the kernel packs; the caller provides the cross-rank barrier before the buffers are read. */
int okp_pack_records_f64(const OkpDecodeTables* tables, int N, int O, int C, int S, long long first_row,
                         double* const* destinations, int n_destinations, void* stream);

/* Ground-truth / training targets for a batch of frames (SURVEY section 8f rank 4). Replaces, per frame, the
 * target construction of the reference's dataset (perception/datasets/video.py): _set_keypoints (:44-53) with the
 * per-map normalisation target / max(target.max(), 0.5) clipped to [0, 1] (:210-211), _compute_centers (:225-242)
 * and _compute_depth (:244-263). keypoints_dev [N,G,Kp,2] float64 (x, y) in TARGET pixels, Kp = 1 +
 * sum(keypoint_config) with each object's centre first (:121-129); depths_dev [N,G,Kp] camera-frame z;
 * n_objects_dev [N] objects present per frame (NULL = G). kernel_size 8, length_scale 2.0, center_radius 4.0 are
 * the reference's constants for its 64x64 targets (:17-20). Outputs: heat_dev [N,C,H,W], centers_dev
 * [N,C-1,2,H,W] (centre - (pixel + 0.5) inside the discs, zero elsewhere), depth_dev [N,C,H,W], float32. */
int okp_rasterise_targets_f32(const double* keypoints_dev, const double* depths_dev, const int32_t* n_objects_dev,
                              int N, int G, int C, int H, int W, const int32_t* keypoint_config, int kernel_size,
                              double length_scale, double center_radius, float* heat_dev, float* centers_dev,
                              float* depth_dev, void* stream);

/* Sparse host -> device transfer of heatmaps for callers that hold them in HOST memory (the reference hands
 * ObjectKeypointPipeline.__call__ CPU tensors, pipeline.py:24-28,184-186). A trained network's heatmaps are almost
 * empty, and a pixel farther than 4 px from every pixel above threshold / 25 can neither be a peak nor beat one in
 * the NMS comparison (its 5x5 box sum stays below the threshold), so replacing such regions by +0 leaves every table
 * bit-identical (proof: csrc/okp_sparse.cuh). okp_host_pack_tiles_f32 runs on the HOST (OpenMP, `threads` <= 0 = all
 * cores): it marks the 4 x 16-pixel tiles of heat_host [maps,H,W] that hold a value above threshold / 25, widens the
 * marks by one tile in every direction and packs the marked tiles into packed_host [capacity_tiles, 64] with
 * tile_ids_host [capacity_tiles] = map * tiles_per_map + tile. scratch_host: okp_host_pack_scratch_bytes() bytes;
 * map_offsets_host: [maps + 1]. *n_tiles_out is the number of marked tiles; if it exceeds capacity_tiles nothing is
 * packed and the caller copies the maps densely (dense inputs, e.g. an untrained network). Only for nms_size 5,
 * box_sum 1 (the reference's configuration) and threshold > 0. */
size_t okp_host_pack_scratch_bytes(int maps, int H, int W);
int okp_host_pack_tiles_f32(const float* heat_host, int maps, int H, int W, float threshold,
                            unsigned char* scratch_host, long long* map_offsets_host, int32_t* tile_ids_host,
                            float* packed_host, long long capacity_tiles, long long* n_tiles_out, int threads);

/* Device side of the sparse transfer: writes the n_tiles packed tiles into heat_dev [maps,H,W], which the caller has
 * zeroed (cudaMemsetAsync) on the same stream. */
int okp_scatter_tiles_f32(const float* packed_dev, const int32_t* tile_ids_dev, long long n_tiles, int maps, int H,
                          int W, float* heat_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OKP_H */
