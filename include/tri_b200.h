/* tri_b200.h -- C ABI of the B200-native batched triangulation engine (libtri_b200.so).
 *
 * This is the drop-in boundary under the reference's C++ `Triangulator` interface
 * (Grzetan/3D-Reconstruction-Triangulation; citations are file:line in that repository).  Plain
 * pointers and sizes only: no C++/torch/OpenCV types.  The C++ adapters in
 * 3d-reconstruction-triangulation_b200/host/ (CudaMatrixTriangulator, CudaRayTriangulator,
 * DroneClassifier) sit on top of these entry points; INTEGRATION.md shows the binding.
 *
 * Every entry point returns a tri_status (0 = ok); tri_last_error() gives the text.  There is no
 * CPU fallback anywhere: without a CUDA device tri_create fails with TRI_ERR_NO_DEVICE.
 */
#ifndef TRI_B200_H
#define TRI_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define TRI_MAX_CAMS 32   /* validity masks are one uint32 per frame (bit c = camera c used)    */
#define TRI_MAX_DETS 15   /* classifier: detections per (camera, frame)                         */
#define TRI_MAX_DRONES 16

typedef enum tri_mode {
  TRI_MATRIX = 0, /* MatrixTriangulator (src/MatrixTriangulator.cpp:3-100), getType() == "matrix" */
  TRI_RAY = 1     /* RayTriangulator    (src/RayTriangulator.cpp:8-107),    getType() == "ray"    */
} tri_mode;

typedef enum tri_status {
  TRI_OK = 0,
  TRI_ERR_DIM = 1,       /* "Every camera should have the same number of points"
                            (MatrixTriangulator.cpp:74-75, RayTriangulator.cpp:56-57)            */
  TRI_ERR_TOO_FEW = 2,   /* "Too few rays are found" (MatrixTriangulator.cpp:93) /
                            "Too few detections are found" (RayTriangulator.cpp:73)              */
  TRI_ERR_ARG = 3,
  TRI_ERR_CUDA = 4,
  TRI_ERR_NO_DEVICE = 5,
  TRI_ERR_CAPACITY = 6   /* a classifier work list overflowed its device buffer                 */
} tri_status;

enum tri_flags {
  TRI_F32 = 1u << 0,              /* matrix / closed-form ray: compute in FP32 (default FP64)    */
  TRI_ALLOW_TOO_FEW = 1u << 1,    /* frames with < 2 views give (0,0,0) and a mask with < 2 bits
                                     instead of TRI_ERR_TOO_FEW (synthetic-batch convention)     */
  TRI_RAY_REFERENCE_LM = 1u << 2, /* ray: follow cv::LMSolver's trajectory exactly (central-
                                     difference Jacobian, DECOMP_EIG solves, 1000-iteration cap,
                                     RayTriangulator.cpp:28-44,100-104); bit-comparable          */
  TRI_RAY_CLOSED_FORM = 1u << 3,  /* ray: the exact minimiser of the reference's (quadratic) objective in one Newton step.
                                     Batch entry points: this IS the default (the flag is accepted and changes nothing).
                                     tri_classify*: opt in to it instead of the reference-LM solves (below)          */
  TRI_PIX_F64 = 1u << 4,          /* pixels are double2 (cv::Point2d) instead of float2          */
  TRI_PIX_U16 = 1u << 5,          /* pixels are ushort2; (0xFFFF,0xFFFF) is the missing marker   */
  TRI_CLS_LAZY = 1u << 7,         /* tri_classify / tri_classify_sequences: the lazy best-first search instead of the candidate
                                     enumeration -- always used above 16 cameras, where the enumeration (like the reference's
                                     own, DroneClassifier.cpp:156-198) is out of reach; same results where both can run   */
  TRI_RAY_ANALYTIC_LM = 1u << 6   /* ray batch: Levenberg-Marquardt with the analytic Jacobian and cv::LMSolver's damping
                                     schedule, register resident (3 iterations; same minimiser as the default)      */
};
/* Ray solver defaults.  tri_triangulate_points*: the closed form -- the reference returns only the point from
 * triangulatePoints (RayTriangulator.cpp:51-81), the objective is quadratic and its LM stops within ~1e-3 mm of this
 * minimiser wherever it converges.  tri_classify*: TRI_RAY_REFERENCE_LM -- the classifier compares the `error` of
 * triangulatePoint against thresholds (DroneClassifier.cpp:185, :209, :243), and cv::LMSolver's last evaluated point
 * (often not converged on 2-view subsets, SURVEY F5) decides differently from the true minimiser; the fast solver
 * there is the explicit TRI_RAY_CLOSED_FORM.                                                                       */

/* What the kernels read of tdr::Camera (src/Camera.h:33-300), filled by the host's Camera class. */
typedef struct tri_camera {
  int32_t width, height;  /* Camera.h:38-39                                                      */
  double fovy_deg;        /* Camera.h:95-97; Triangulator.cpp:33-34 reads it                     */
  double P[12];           /* cameraPerspectiveMatrix, row-major 3x4 (Camera.h:159-161)           */
  double position[3];     /* "tvec" = world position (utils.cpp:101, Triangulator.cpp:50-54)     */
  double quat[4];         /* "rquat" (w,i,j,k) as stored, not normalised (Triangulator.cpp:15-25)*/
} tri_camera;

/* Optional per-frame outputs of the batch entry points; any pointer may be NULL except that at
 * least one of xyz_f32 / xyz_f64 must be set. */
typedef struct tri_batch_out {
  float* xyz_f32;    /* [n_frames][3] packed, 12 B per point                                     */
  double* xyz_f64;   /* [n_frames][3]                                                            */
  uint32_t* mask;    /* bit c set <=> camera c had x != -1 && y != -1 (MatrixTriangulator.cpp:86)*/
  double* err;       /* the `error` of triangulatePoint (MatrixTriangulator.cpp:55-59 /
                        RayTriangulator.cpp:26)                                                  */
  int32_t* iters;    /* ray: LM iterations                                                       */
} tri_batch_out;

typedef struct tri_classify_stats {
  int64_t nodes, solves, leaves, lm_iters, phase1, phase2, ties, max_frontier;
  int64_t enumerate_us, link_us; /* device time (CUDA events) of candidate generation / of the sequential linking pass */
} tri_classify_stats;

typedef struct tri_engine tri_engine;

int tri_version(void);
const char* tri_last_error(void);
int tri_device_count(void);

/* One engine = one GPU + the camera rig (replaces `new MatrixTriangulator(cameras)` /
 * `new RayTriangulator(cameras)`, src/main.cpp:54-63; constructors MatrixTriangulator.h:19,
 * RayTriangulator.h:34).  The camera constants are copied. */
int tri_create(int n_cams, const tri_camera* cams, int device, tri_engine** out);
void tri_destroy(tri_engine* e);
int tri_engine_device(const tri_engine* e);
int tri_engine_cameras(const tri_engine* e);
/* number of kernels this engine has launched so far (bench.py's gpu_launches) */
int64_t tri_kernel_launches(const tri_engine* e);

/* Triangulator::triangulatePoints (Triangulator.h:51-52; MatrixTriangulator.cpp:70-100,
 * RayTriangulator.cpp:51-81), HOST buffers.  xy is structure-of-arrays [n_point_cams][n_frames]
 * pixel pairs, camera rows `cam_stride` pixels apart (>= n_frames), (-1,-1) = no detection.
 * Matrix mode uses min(n_point_cams, n_cams) rows (MatrixTriangulator.cpp:84); ray mode requires
 * n_point_cams <= n_cams (the reference reads out of bounds otherwise, RayTriangulator.cpp:65-69).
 * Frames stream through the GPU in chunks (H2D copy, kernel and D2H copy overlapped).
 * On TRI_ERR_TOO_FEW *first_bad_frame (may be NULL) is the first frame with < 2 views. */
int tri_triangulate_points(tri_engine* e, int mode, unsigned flags, const void* xy, int n_point_cams,
                           int64_t n_frames, int64_t cam_stride, const tri_batch_out* out,
                           int64_t* first_bad_frame);

/* Outlier-robust matrix-mode batch (an extension: the reference has no such call).  Same pixel layout, camera rows
 * (min(n_point_cams, n_cams)), missing-view test and too-few handling as tri_triangulate_points in TRI_MATRIX mode.
 * Per frame with valid views V (|V| >= 2): every pair i < j of V gives the two-view DLT X_ij, usable if its projective
 * depth w_c = P_c[8..10].X + P_c[11] is > 0 on both cameras; its inliers are the views c of V with w_c(X_ij) > 0 and
 * pixel reprojection error r_c <= max_reproj_px; the winner has the most inliers (>= 2), then the smallest sum of r_c^2
 * over them, then the first pair in (i, j) order; the result is the DLT over the winner's inlier set I.  One consensus
 * round, one refit, FP64 (FP32 under TRI_F32).  The fields of tri_batch_out mean, for these two calls:
 *   xyz_f32 / xyz_f64  the refitted point; (0,0,0) when no hypothesis has 2 inliers (not an error)
 *   mask               the inlier set I (0 when there is no consensus; the < 2 valid bits on a too-few frame)
 *   err                RMS pixel reprojection error of the point over I, sqrt(mean r_c^2); NaN without consensus,
 *                      0 on a too-few frame
 *   iters              must be NULL
 * Flags: TRI_F32, TRI_PIX_F64, TRI_PIX_U16, TRI_ALLOW_TOO_FEW; anything else, max_reproj_px <= 0 or NaN, or a
 * non-NULL iters returns TRI_ERR_ARG.  HOST buffers, streamed in chunks like tri_triangulate_points. */
int tri_triangulate_points_robust(tri_engine* e, unsigned flags, double max_reproj_px, const void* xy, int n_point_cams,
                                  int64_t n_frames, int64_t cam_stride, const tri_batch_out* out, int64_t* first_bad_frame);
/* The same with DEVICE buffers, asynchronous on `stream`; too-few frames are latched for tri_device_status. */
int tri_triangulate_points_robust_device(tri_engine* e, unsigned flags, double max_reproj_px, const void* d_xy,
                                         int n_point_cams, int64_t n_frames, int64_t cam_stride,
                                         const tri_batch_out* d_out, void* stream);

/* The same batch sharded over several engines (one per GPU of the box) from ONE host process: frames
 * are independent, so engine g takes the contiguous range [g*N/G, (g+1)*N/G) and the shards run
 * concurrently (one host thread and one copy/compute pipeline per GPU); results land in the caller's
 * host buffers in frame order, no collective needed.  All engines must hold the same rig. */
int tri_triangulate_points_multi(tri_engine* const* engines, int n_engines, int mode, unsigned flags,
                                 const void* xy, int n_point_cams, int64_t n_frames, int64_t cam_stride,
                                 const tri_batch_out* out, int64_t* first_bad_frame);

/* Same with DEVICE buffers, asynchronous on `stream` (a cudaStream_t, NULL = default stream).
 * The too-few-views condition is latched on the device; tri_device_status collects it. */
int tri_triangulate_points_device(tri_engine* e, int mode, unsigned flags, const void* d_xy,
                                  int n_point_cams, int64_t n_frames, int64_t cam_stride,
                                  const tri_batch_out* d_out, void* stream);
/* Fused gather over NVLink: the device entry point writes its points with plain stores, so `d_out->xyz_f32`
 * may point into ANOTHER GPU's memory (a peer-mapped or CUDA-IPC-opened buffer, e.g. rank 0's result array at
 * this rank's frame offset): the gather then happens inside the kernel's epilogue, tile by tile, instead of as a
 * separate collective.  This enables the peer mapping from the engine's GPU to `peer_device` once. */
int tri_enable_peer_access(tri_engine* e, int peer_device);
/* CUDA IPC for that: export a buffer obtained from tri_device_alloc (64-byte handle to hand to the other
 * processes of the box), open such a handle on this engine's GPU (peer access is enabled lazily), close it. */
int tri_ipc_export(tri_engine* e, void* d_ptr, unsigned char handle[64]);
int tri_ipc_open(tri_engine* e, const unsigned char handle[64], void** d_ptr);
int tri_ipc_close(tri_engine* e, void* d_ptr);
int tri_copy_device(tri_engine* e, void* d_dst, const void* d_src, uint64_t bytes);

/* Synchronises `stream`, returns TRI_ERR_TOO_FEW if a frame was latched since the last call. */
int tri_device_status(tri_engine* e, void* stream, int64_t* first_bad_frame);

/* Triangulator::triangulatePoint (Triangulator.h:46-47; MatrixTriangulator.cpp:3-62,
 * RayTriangulator.cpp:83-107) for many (camera subset, pixels) items at once; HOST buffers.
 * Item i uses cam_idx/xy entries [item_offsets[i], item_offsets[i+1]).  xyz [n_items][3],
 * err [n_items], iters [n_items] (may be NULL). */
int tri_triangulate_subsets(tri_engine* e, int mode, unsigned flags, int64_t n_items,
                            const int32_t* item_offsets, const int32_t* cam_idx, const double* xy,
                            double* xyz, double* err, int32_t* iters);

/* Triangulator::getDistFromRay (Triangulator.h:58, Triangulator.cpp:57-61), batched; HOST buffers.
 * out[i] = distance of points[i] to the ray of pixel xy[i] on camera cam_idx[i]. */
int tri_dist_from_ray(tri_engine* e, int64_t n, const int32_t* cam_idx, const double* xy,
                      const double* points, double* out);

/* DroneClassifier::classifyDrones (DroneClassifier.cpp:96-154); HOST buffers.  Up to 16 cameras the candidate combinations
 * are enumerated frame-parallel and then linked; 17..32 cameras (or TRI_CLS_LAZY) run the lazy best-first search.
 * Detections in CSR form: det_offsets[cam*(n_frames+1)+f] indexes dets_xy pairs ordered
 * [cam][frame][det].  out_paths [n_drones][n_frames][3]; out_assign [n_drones][n_frames][n_cams]
 * combination indices (0 = camera unused, k = detection k-1; -1 = the path got no point in that
 * frame); out_phase [n_drones][n_frames]: 0 none, 1 tracking (:119-135), 2 (re)initialisation
 * (:140-143).  out_assign / out_phase / stats may be NULL. */
int tri_classify(tri_engine* e, int mode, unsigned flags, int n_drones, const int32_t* det_offsets,
                 const double* dets_xy, int n_frames, double* out_paths, int8_t* out_assign,
                 uint8_t* out_phase, tri_classify_stats* stats);

/* Many independent sequences (recordings) in one call: sequence q holds the frames [seq_bounds[q], seq_bounds[q+1]) of
 * the CSR (seq_bounds[0] = 0, seq_bounds[n_seq] = n_frames).  Candidate generation runs over all frames at once and
 * every sequence is linked by its own warp, so the sequential part of classifyDrones (DroneClassifier.cpp:112-144)
 * costs the longest sequence, not the sum.  Outputs as in tri_classify ([n_drones][n_frames] rows); each sequence's
 * result equals tri_classify on that sequence alone. */
int tri_classify_sequences(tri_engine* e, int mode, unsigned flags, int n_drones, int n_seq, const int32_t* seq_bounds,
                           const int32_t* det_offsets, const double* dets_xy, int n_frames, double* out_paths,
                           int8_t* out_assign, uint8_t* out_phase, tri_classify_stats* stats);

/* The same over a frame-sharded sequence (one engine per GPU; SURVEY 8e): candidate generation is independent
 * per frame (fillCombinationQueue, DroneClassifier.cpp:156-198), linking is sequential (classifyDrones' path
 * state, :119-135, :269-297).  tri_classify_begin enumerates this engine's contiguous shard of the sequence and
 * keeps the candidates on the device; tri_classify_finish links the shard starting from `state_in` -- the opaque
 * tri_classify_state_bytes() blob tri_classify_finish returned for the PREVIOUS shard (NULL = start of the
 * sequence) -- and writes the state after the shard's last frame to `state_out` (may be NULL).  Outputs as in
 * tri_classify, for the shard's frames; concatenated over the shards they equal tri_classify on the whole
 * sequence bit for bit. */
int tri_classify_state_bytes(void);
int tri_classify_begin(tri_engine* e, int mode, unsigned flags, int n_drones, const int32_t* det_offsets,
                       const double* dets_xy, int n_frames);
int tri_classify_finish(tri_engine* e, const void* state_in, void* state_out, double* out_paths, int8_t* out_assign,
                        uint8_t* out_phase, tri_classify_stats* stats);
/* One host process, one engine per GPU: begin on every engine concurrently, finish in order.  Arguments and
 * results as tri_classify. */
int tri_classify_multi(tri_engine* const* engines, int n_engines, int mode, unsigned flags, int n_drones,
                       const int32_t* det_offsets, const double* dets_xy, int n_frames, double* out_paths,
                       int8_t* out_assign, uint8_t* out_phase, tri_classify_stats* stats);

/* Memory helpers so a host without CUDA headers can own pinned / device buffers. */
int tri_host_alloc(void** p, uint64_t bytes);   /* page-locked */
int tri_host_free(void* p);
int tri_device_alloc(tri_engine* e, void** p, uint64_t bytes);
int tri_device_free(tri_engine* e, void* p);
int tri_copy_to_device(tri_engine* e, void* d_dst, const void* h_src, uint64_t bytes);
int tri_copy_to_host(tri_engine* e, void* h_dst, const void* d_src, uint64_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* TRI_B200_H */
