/*
 * bpc_b200.h -- C ABI of libbpc_b200.so: the B200 (sm_100a) implementation of the bpc_baseline
 * multi-camera match + ROI-crop hot path.
 *
 * The reference (yatpor/bpc_baseline) is pure Python and has no FFI layer; its boundary for this
 * path is the Python function surface of bpc/inference/{epipolar_matching,process_pose}.py,
 * bpc/inference/utils/{camera_utils,triangulation}.py and bpc/utils/data_utils.py.  Each entry
 * point below names the reference function (file:line) it replaces; INTEGRATION.md shows the
 * ctypes binding a maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless marked "host"; buffers are dense, row-major;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - calls are asynchronous and stream-ordered: no allocation, no synchronisation, no host
 *     read-back inside the library; workspaces are supplied by the caller;
 *   - return value: BPC_OK, a negative BPC_E* argument error, or a positive cudaError_t.
 *
 * Batched scene layout (S scenes, 3 cameras, at most Dmax detections per camera):
 *   Ks      float   [S][3][3][3]     intrinsics                      camera_utils.py:16
 *   RTs     double  [S][3][4][4]     world->camera, f32 values widened, data_utils.py:383-387
 *   centers double  [S][3][Dmax][2]  detection centres 'bb_center'   process_pose.py:135-136
 *   boxes   int32   [S][3][Dmax][4]  (x1,y1,x2,y2) 'bbox'            process_pose.py:134
 *   counts  int32   [S][3]           detections per camera (ragged N, M, P)
 */
#ifndef BPC_B200_H
#define BPC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BPC_ABI_VERSION 2

enum {
    BPC_OK = 0,
    BPC_EINVAL = -1,     /* bad size / null pointer / unsupported value */
    BPC_EALIGN = -2,     /* pointer not aligned as documented */
    BPC_EWORKSPACE = -3, /* workspace too small */
    BPC_ETOOBIG = -4,    /* problem exceeds a documented limit (Dmax, ROI width) */
    BPC_EUNSUPPORTED = -5 /* the variant does not exist for this configuration (see the entry point's comment) */
};

/* per-scene status values of the `n` output of the matchers (any negative n: the scene has no matches) */
#define BPC_N_INFEASIBLE (-1)   /* NaN / -inf / all-infinite costs: scipy.optimize.linear_sum_assignment raises ValueError */
#define BPC_N_OVERFLOW (-2)     /* a camera's count exceeds Dmax (e.g. the overflow count of bpc_detections_from_yolo) */

/* limits */
#define BPC_MAX_DET 2048        /* Dmax <= 2048 detections per camera; a scene stays in shared memory up to Dmax ~ 550,
                                   larger scenes keep their state in the caller's workspace (bpc_match_workspace_bytes) */
#define BPC_MAX_ROI_WIDTH 8192  /* widest source box the crop kernel stages in shared memory */
#define BPC_MAX_TARGET 1024     /* crop target size T <= 1024 (one thread per output column in the generic kernel) */

int bpc_abi_version(void);
/* Static string for a code returned by any entry point (host pointer, never freed). */
const char* bpc_error_string(int code);

/* ------------------------------------------------------------------------------------------
 * a1. Fundamental matrices F12, F13, F23 of every scene.
 * Replaces compute_fundamental_matrix, bpc/inference/utils/camera_utils.py:23-46, as called
 * three times by PoseEstimator._match, bpc/inference/process_pose.py:154-159.
 *   F  double [S][3][3][3]   (pair order 12, 13, 23; F_ab maps a cam-a point to its cam-b line)
 */
int bpc_fundamental(const float* Ks, const double* RTs, int S, double* F, void* stream);

/* ------------------------------------------------------------------------------------------
 * a2-a4. Materialised N x M x P cost tensor (small D / tests; the matcher never builds it).
 * Replaces compute_cost_matrix, bpc/inference/epipolar_matching.py:83-98 (epipolar_error :5-28,
 * epipolar_error_full :73-81).
 *   F     double [S][3][3][3]   from bpc_fundamental (or any caller-supplied F12,F13,F23)
 *   cost  float  [S][Dmax][Dmax][Dmax]; entries beyond (N,M,P) of a scene are left untouched
 */
int bpc_cost_tensor(const double* F, const double* centers, const int32_t* counts, int S, int Dmax,
                    float* cost, void* stream);

/* ------------------------------------------------------------------------------------------
 * a5. Thresholded rectangular assignment on an explicit cost tensor.
 * Replaces match_objects, bpc/inference/epipolar_matching.py:100-116 (scipy
 * linear_sum_assignment on cost.reshape(N*M, P), keep cost < threshold, ascending r = i*M+j).
 *   cost       float [S][N][M][P]          dense, same N, M, P for the whole batch
 *   idx        int32 [S][Kmax][3]          (i, j, k) per kept match, ascending r, -1 padded
 *   n          int32 [S]                   kept matches per scene
 *   n          = BPC_N_INFEASIBLE where SciPy raises (any NaN or -inf entry, or no feasible assignment)
 *   Kmax       = min(N*M, P)
 * The assignment state (O(rows) words + one bit per column) lives in shared memory: BPC_ETOOBIG beyond that.
 */
int bpc_match_objects(const float* cost, int S, int N, int M, int P, float threshold,
                      int32_t* idx, int32_t* n, void* stream);

/* ------------------------------------------------------------------------------------------
 * a1-a10. The whole geometry path of PoseEstimator._match, bpc/inference/process_pose.py:144-188,
 * for S independent scenes: fundamental matrices, virtual cost tensor, assignment, threshold,
 * stable sort by cost (:183), DLT triangulation of every match (PosePrediction :79-94,
 * triangulate_multi_view epipolar_matching.py:118-127) and per-view reprojection error
 * (compute_reprojection_error, bpc/inference/utils/triangulation.py:14-18).
 *   threshold  compared as float32 against the float32 cost (epipolar_matching.py:110-111)
 *   has_reproj_thresh, reproj_thresh
 *              optional reprojection-error filter: with has_reproj_thresh != 0 a match is dropped when the error of ANY
 *              view exceeds reproj_thresh pixels (error > reproj_thresh: an equal or NaN error is kept); survivors keep
 *              their (cost, r) order, n is updated, the tail re-padded.
 *              The reference has the helper but no call site that filters (SURVEY.md F7), so 0 = reference behaviour;
 *              needs reproj != NULL.
 *   Kmax       = Dmax
 *   idx    int32  [S][Kmax][3]  matches sorted by (cost, r); -1 padded
 *   n      int32  [S]           matches per scene (0 if any camera has no detection, :161-163; BPC_N_INFEASIBLE where
 *                               SciPy raises: a NaN cost, e.g. from a NaN or infinite centre, or no feasible assignment;
 *                               BPC_N_OVERFLOW if a count exceeds Dmax -- never a silent empty result)
 *   cost   float  [S][Kmax]     cost of each match (NaN padded)
 *   X      double [S][Kmax][3]  triangulated points (NaN padded)
 *   reproj double [S][Kmax][3]  reprojection error per view, pixels (NaN padded); may be NULL
 *   F      double [S][3][3][3]  fundamental matrices; may be NULL
 * Workspace: bpc_match_workspace_bytes(S, Dmax) bytes, 16-byte aligned: 0 while a scene fits shared memory (Dmax up to
 * ~550), else one state block per resident CTA (the kernel then walks the scenes with a fixed grid).
 */
size_t bpc_match_workspace_bytes(int S, int Dmax);
int bpc_match_triangulate(const float* Ks, const double* RTs, const double* centers, const int32_t* counts,
                          int S, int Dmax, float threshold, int has_reproj_thresh, double reproj_thresh,
                          int32_t* idx, int32_t* n, float* cost, double* X, double* reproj, double* F,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Pose records for the final multi-GPU gather (SURVEY.md 8e): the valid match slots of every scene, compacted in
 * scene order, native dtypes, 64 bytes each:  idx int32 x3 | cost float | X double x3 | reproj double x3.
 *   buf = | total int32, S int32, Kmax int32, 0 | n int32 [S], padded to 16 bytes | records ... |
 *   scene_offset int32 [S+1]  exclusive prefix sum of offset_div * max(n, 0); bpc_build_rois' output with offset_div = 3
 *   reproj       may be NULL (NaN is written)
 *   buf          bpc_pack_records_bytes(S, Kmax) bytes (capacity S*Kmax records), 16-byte aligned
 */
size_t bpc_pack_records_bytes(int S, int Kmax);
int bpc_pack_records(const int32_t* idx, const int32_t* n, const float* cost, const double* X, const double* reproj,
                     const int32_t* scene_offset, int offset_div, int S, int Kmax, void* buf, void* stream);

/* ------------------------------------------------------------------------------------------
 * a8. Stand-alone DLT triangulation.  Replaces triangulate_multi_view,
 * bpc/inference/epipolar_matching.py:118-127 (= utils/triangulation.py:3-12) for 3 views.
 *   P    double [n][3][3][4]   projection matrices
 *   pts  double [n][3][2]      image points
 *   X    double [n][3]
 * a9. Reprojection error, bpc/inference/utils/triangulation.py:14-18.
 *   err  double [n][3]
 */
int bpc_triangulate(const double* P, const double* pts, int n, double* X, void* stream);
/* a7. Projection matrices P = K (float32) @ RT[:3] (float64), bpc/inference/process_pose.py:88-92.
 *   K float [n][3][3], RT double [n][4][4]  ->  P double [n][3][4] */
int bpc_projection(const float* K, const double* RT, int n, double* P, void* stream);
int bpc_reprojection_error(const double* P, const double* X, const double* pts, int n, double* err, void* stream);

/* ------------------------------------------------------------------------------------------
 * a2, a3. Scalar distances for n independent inputs (the reference's per-pair functions).
 * bpc_epipolar_error      replaces epipolar_error(pt1, pt2, F), epipolar_matching.py:5-28
 *   F double [n][3][3], pt1 / pt2 double [n][2]  ->  e double [n]
 * bpc_epipolar_error_full replaces epipolar_error_full(pt1, pt2, pt3, F12, F13, F23), :73-81
 *   F double [n][3][3][3] (12, 13, 23), pts double [n][3][2]  ->  e double [n]
 * bpc_triangulate_views   triangulate_multi_view for V views (2 <= V <= 8), :118-127
 *   P double [n][V][3][4], pts double [n][V][2]  ->  X double [n][3]
 */
int bpc_epipolar_error(const double* F, const double* pt1, const double* pt2, int n, double* e, void* stream);
int bpc_epipolar_error_full(const double* F, const double* pts, int n, double* e, void* stream);
int bpc_triangulate_views(const double* P, const double* pts, int n, int V, double* X, void* stream);

/* Centres from integer boxes: cx = 0.5*(x1+x2), cy = 0.5*(y1+y2), process_pose.py:134-136. */
int bpc_box_centers(const int32_t* boxes, int count, double* centers, void* stream);

/* Detector post-processing (producer side of the path, SURVEY.md 8f rank 2): class / confidence filter,
 * int() truncation of the box, centre -- the loop of PoseEstimator._detect, bpc/inference/process_pose.py:123-141,
 * producing the device-resident detection tensors the matcher consumes.
 *   xyxy float [SC][Nraw][4] (16-byte aligned), conf / cls float [SC][Nraw], nraw int32 [SC]; SC = scenes * cameras
 *   keeps cls == 0 && conf >= conf_thresh, in order; boxes int32 [SC][Dmax][4], centers double [SC][Dmax][2]
 *   counts int32 [SC] = number kept (entries beyond Dmax are dropped; counts > Dmax signals the overflow, which
 *                       bpc_match_triangulate reports as n = BPC_N_OVERFLOW for that scene)
 */
int bpc_detections_from_yolo(const float* xyxy, const float* conf, const float* cls, const int32_t* nraw, int SC, int Nraw,
                             float conf_thresh, int Dmax, int32_t* boxes, double* centers, int32_t* counts, void* stream);

/* ------------------------------------------------------------------------------------------
 * ROI records for the crop kernel from the matcher's output: 3 per match in (scene, match, view)
 * order, rois int32 [R][5] = (image index, x1, y1, x2, y2).  Mirrors the loops of
 * PoseEstimator._estimate_rotation, process_pose.py:195-201.
 *   image_of_scene int32 [S][3]     index of each view's image in the image pool
 *   scene_offset   int32 [S + 1]    exclusive prefix sum of 3*n (output; scene_offset[S] = R)
 *   rois           int32 [S*Kmax*3][5] capacity
 */
int bpc_build_rois(const int32_t* boxes, const int32_t* idx, const int32_t* n, const int32_t* image_of_scene,
                   int S, int Dmax, int Kmax, int32_t* scene_offset, int32_t* rois, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training-side ROI records (SURVEY 8f rank 3): the crop windows BOPSingleObjDataset.__getitem__
 * takes, bpc/utils/data_utils.py:243-271, as rois int32 [n][5] for bpc_roi_crop (swap_rb = 0: the
 * dataset keeps the BGR order, :249-252).
 *   xywh   int32 [n][4]   bbox_visib (x, y, w, h)                               :242
 *   image  int32 [n]      index of each sample's image in the pool; NULL = 0
 *   scale  double [n]     NULL = the original crop bgr[y:y+h, x:x+w] (:246); else the augmented one:
 *                         scale_factor of :257, aug_w = int(round(w * scale)) (half-to-even), clamps of :264-267
 *   shift  int32 [n][2]   (shift_x, shift_y) of :262-263; NULL = 0.  The random draws stay on the host
 *                         (Python's `random` stream is the reference's); this only applies them.
 *   W, H   image size
 */
int bpc_train_rois(const int32_t* xywh, const int32_t* image, const double* scale, const int32_t* shift, int n,
                   int W, int H, int32_t* rois, void* stream);

/* ------------------------------------------------------------------------------------------
 * a11 + a12. Crop -> letterbox (INTER_AREA) -> colour order -> /255 -> normalise, for R ROIs.
 * Replaces letterbox_preserving_aspect_ratio, bpc/utils/data_utils.py:34-44, and the inline
 * transform of PoseEstimator._estimate_rotation, bpc/inference/process_pose.py:199-209
 * (training twin: data_utils.py:243-252,282 = swap_rb 0).
 *   images   uint8 [B][H][W][3]   BGR, 16-byte aligned base
 *   rois     int32 [R][5]         (image, x1, y1, x2, y2), 0 <= x1 < x2 <= W, 0 <= y1 < y2 <= H
 *   n_rois_dev  optional device int32 holding the TOTAL number of valid ROIs of the batch the
 *               records belong to (e.g. scene_offset[S] of bpc_build_rois); NULL = all R are valid
 *   roi_first   index, within that batch, of rois[0] (chunked processing into a reusable `out`):
 *               record r is processed iff roi_first + r < *n_rois_dev
 *   T        target size (reference default 256)
 *   fill     host uint8[3], letterbox colour in source channel order
 *   swap_rb  1 = BGR->RGB as cv2.cvtColor(COLOR_BGR2RGB) at process_pose.py:206
 *   lut      float [3][256]: lut[c][v] = normalised value of byte v in OUTPUT channel c
 *   out      float [R][3][T][T]   (16-byte aligned)
 *   status   optional int32 [R]: 0 ok, 1 = ROI rejected (empty box, resized side < 1, out of
 *            image, wider than BPC_MAX_ROI_WIDTH); a rejected ROI's output is all fill colour
 *   workspace   bpc_roi_crop_workspace_bytes(R, T) bytes of device scratch (16-byte aligned): per-ROI
 *               geometry records, tap descriptors and the list of ROIs taking the generic path
 * bpc_roi_crop_u8 writes the uint8 letterboxed image itself, uint8 [R][T][T][3] in source channel
 * order -- exactly what letterbox_preserving_aspect_ratio returns.
 */
size_t bpc_roi_crop_workspace_bytes(int R, int T);
int bpc_roi_crop(const uint8_t* images, int B, int H, int W, const int32_t* rois, int R,
                 const int32_t* n_rois_dev, int roi_first, int T, const uint8_t* fill, int swap_rb,
                 const float* lut, float* out, int32_t* status,
                 void* workspace, size_t workspace_bytes, void* stream);
int bpc_roi_crop_u8(const uint8_t* images, int B, int H, int W, const int32_t* rois, int R,
                    const int32_t* n_rois_dev, int roi_first, int T, const uint8_t* fill,
                    uint8_t* out, int32_t* status,
                    void* workspace, size_t workspace_bytes, void* stream);
/* bpc_roi_crop_bf16: the network-input variant for a bf16 tensor-core pose head (process_pose.py:210-212 moves the float32
 * tensor to the GPU and runs SimplePoseNet on it): every value of bpc_roi_crop's float32 tensor rounded to bfloat16
 * (round-to-nearest-even) and stored channels-last, out = bfloat16 [R][T][T][3] (16-byte aligned) -- half the output bytes,
 * no layout pass before the first convolution.  Exists on the 2-D-TMA path only: image row pitch W*3 a multiple of 16 bytes
 * and >= 1600, T <= 256; otherwise BPC_EUNSUPPORTED (use bpc_roi_crop). */
int bpc_roi_crop_bf16(const uint8_t* images, int B, int H, int W, const int32_t* rois, int R,
                      const int32_t* n_rois_dev, int roi_first, int T, const uint8_t* fill, int swap_rb,
                      const float* lut, void* out, int32_t* status,
                      void* workspace, size_t workspace_bytes, void* stream);
/* lut[c][v] = (v/255 - mean[c]) / std[c] in float32 with true divisions, as torchvision's
 * to_tensor (.div(255)) + normalize (.sub_(mean).div_(std)); process_pose.py:207-209. */
int bpc_normalise_lut(const float* mean_host3, const float* std_host3, float* lut, void* stream);

/* ---- crop gather (receiver side) --------------------------------------------------------------
 * The colour swap + to_tensor + normalize tail of process_pose.py:206-209 applied to uint8
 * letterboxed crops [count][T][T][3] (the output of bpc_roi_crop_u8) that live in up to 16 source
 * buffers, concatenated in source order into out float32 [sum(counts)][3][T][T]; bit-identical to
 * what bpc_roi_crop writes for the same ROIs.  `srcs` and `counts` are HOST arrays of n_src device
 * pointers / crop counts.  A source pointer may be another GPU's buffer mapped into this process
 * (e.g. torch symmetric memory: a VMM mapping with access for this device): the
 * kernel then pulls the bytes over NVLink while converting -- the gather and the arithmetic are one
 * kernel and the wire carries 1 byte per sample instead of 4.  Fast path: T % 4 == 0 and 16-byte
 * aligned pointers; anything else takes a scalar kernel. */
int bpc_crops_normalise(const uint8_t* const* srcs, const int32_t* counts, int n_src, int T, int swap_rb,
                        const float* lut, float* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training-side ColorJitter (SURVEY 8f rank 3): torchvision.transforms.ColorJitter on
 * Image.fromarray(canvas), then to_tensor + normalize -- what BOPSingleObjDataset.__getitem__ does
 * with the jittered canvas (bpc/utils/data_utils.py), bit-exact with Pillow's arithmetic.  The
 * random draws stay on the host (torch's RNG stream, ColorJitter.get_params); this only applies them.
 *   in       uint8 [n][T][T][3]   e.g. the output of bpc_roi_crop_u8; stored channel 0 is PIL's R
 *   order    int32 [n][4]         op ids in application order: 0 brightness, 1 contrast, 2 saturation,
 *                                 3 hue, -1 = no op; each id at most once per crop (not checked: a repeated
 *                                 contrast would reuse the first one's mean)
 *   factors  float [n][4]         (brightness, contrast, saturation, hue) as float32 values; entries of
 *                                 ops absent from `order` are ignored (any value, NaN included)
 *   swap_rb, lut                  as bpc_roi_crop (the dataset uses swap_rb = 0)
 *   out      float [n][3][T][T]
 * 1 <= T <= BPC_MAX_TARGET; no workspace.  Fast path: T % 4 == 0 and 16-byte aligned in / out.
 */
int bpc_color_jitter(const uint8_t* in, int n, int T, const int32_t* order, const float* factors, int swap_rb,
                     const float* lut, float* out, void* stream);

/* Number of kernel launches issued by this library since load (all entry points). */
unsigned long long bpc_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* BPC_B200_H */
