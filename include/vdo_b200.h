/*
 * vdo_b200.h -- C ABI of the B200-native VDO-SLAM hot path (libvdo_b200.so).
 *
 * The reference (halajun/VDO_SLAM) has no FFI layer: its hot path is plain C++ inside libObjSLAM.so.
 * Each entry point below names the reference interface it replaces (paths relative to the reference root;
 * g2o/ = dependencies/g2o/g2o/).  Host wrappers with the reference's own C++ signatures
 * (VDO_SLAM::Optimizer, ORBextractor, ...) sit above this ABI; see INTEGRATION.md.
 *
 * Conventions
 *   - plain pointers + sizes, caller-allocated outputs, int status return (0 = VDO_OK, <0 = error;
 *     vdo_last_error() gives the text).  No exceptions cross the boundary, nothing calls exit().
 *   - every pointer is a HOST pointer unless the parameter name ends in _dev.
 *   - an SE(3) value ("iso") is 12 doubles: rotation row-major (9) then translation (3) -- the memory
 *     image of g2o's Isometry3 estimate (g2o/types/vertex_se3.h:50) without Eigen's column-major packing.
 *   - there is NO CPU fallback: every compute entry point fails with VDO_ERR_CUDA when no sm_100 device
 *     is usable.
 */
#ifndef VDO_B200_H
#define VDO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VDO_OK 0
#define VDO_ERR_CUDA (-1)        /* CUDA runtime / no device */
#define VDO_ERR_ARG (-2)         /* bad argument */
#define VDO_ERR_UNSUPPORTED (-3) /* graph shape outside what the reference's optimisers build */
#define VDO_ERR_STATE (-4)       /* call order violated */
#define VDO_ERR_NCCL (-5)

typedef struct vdo_ctx vdo_ctx;     /* one per VDO_SLAM::System (src/System.cc:22-48): device, stream, arenas */
typedef struct vdo_graph vdo_graph; /* one per g2o::SparseOptimizer instance of the batch optimisers */

int vdo_ctx_create(int device, vdo_ctx **out);
void vdo_ctx_destroy(vdo_ctx *ctx);
const char *vdo_last_error(const vdo_ctx *ctx);
/* cudaStream_t of the context as an integer handle (so torch / callers can order work against it) */
uint64_t vdo_ctx_stream(const vdo_ctx *ctx);

/* Multi-GPU (one process per GPU).  The batch graph shards by tracklet: after vdo_ctx_init_comm, vdo_graph_finalize keeps
 * the tracklets of this rank only (round-robin), the se3 state is replicated, and partial se3-side sums are all-reduced
 * over NCCL (H_pp/b_p once per linearisation, the 6C-vector S*p once per PCG iteration, chi2/scale once per LM trial).
 * rank 0 calls vdo_nccl_unique_id and ships the 128 bytes to the other ranks (e.g. torch.distributed broadcast). */
int vdo_nccl_unique_id(char *out128);
int vdo_ctx_init_comm(vdo_ctx *ctx, int rank, int world, const char *id128);

/* ------------------------------------------------------------------------------------------------
 * Batch factor-graph optimisation.  Replaces the g2o::SparseOptimizer + OptimizationAlgorithmLevenberg +
 * BlockSolverX + LinearSolverCSparse stack as driven by Optimizer::FullBatchOptimization
 * (src/Optimizer.cc:1232-2175) and Optimizer::PartialBatchOptimization (src/Optimizer.cc:42-1230).
 * ------------------------------------------------------------------------------------------------ */

/* new g2o::SparseOptimizer (src/Optimizer.cc:1312-1323, :172-183) */
int vdo_graph_create(vdo_ctx *ctx, vdo_graph **out);
void vdo_graph_destroy(vdo_graph *g);

/* optimizer.addVertex(VertexSE3 / VertexPointXYZ) with setEstimate (src/Optimizer.cc:1359-1363, 1412-1416,
 * 1571-1582).  se3: n_se3 x 12 iso (camera poses and object motions share one index space), pt: n_pt x 3. */
int vdo_graph_set_vertices(vdo_graph *g, int n_se3, const double *se3, int n_pt, const double *pt);

/* EdgeSE3Prior, identity offset parameter, information = w * I6, no kernel (src/Optimizer.cc:1364-1373;
 * g2o/types/edge_se3_prior.cpp:89-102).  v: n se3 indices, Z: n x 12 iso, w: n */
int vdo_graph_add_edges_se3_prior(vdo_graph *g, int n, const int *v, const double *Z, const double *w);

/* EdgeSE3 (odometry and motion-smoothness edges; src/Optimizer.cc:1383-1399, 1596-1623;
 * g2o/types/edge_se3.cpp:77-104).  ij: n x 2 se3 indices, Z: n x 12, information = w * I6,
 * Huber delta (<= 0: no robust kernel). */
int vdo_graph_add_edges_se3(vdo_graph *g, int n, const int *ij, const double *Z, const double *w, const double *delta);

/* EdgeSE3PointXYZ, identity offset (src/Optimizer.cc:1421-1435; g2o/types/edge_se3_pointxyz.cpp:99-140).
 * cp: n x 2 (se3 index, point index), z: n x 3 measured point in the camera frame, information = w * I3 */
int vdo_graph_add_edges_se3_pointxyz(vdo_graph *g, int n, const int *cp, const double *z, const double *w, const double *delta);

/* LandmarkMotionTernaryEdge, measurement 0 (src/Optimizer.cc:1724-1741; g2o/types/types_dyn_slam3d.cpp:53-85).
 * pph: n x 3 (point p1, point p2, motion se3 index), information = w * I3 */
int vdo_graph_add_edges_landmark_motion(vdo_graph *g, int n, const int *pph, const double *w, const double *delta);

/* optimizer.initializeOptimization() + BlockSolver::buildStructure (src/Optimizer.cc:1768;
 * g2o/core/block_solver.hpp:142-295): orders landmarks by tracklet, builds the edge streams, uploads to HBM. */
int vdo_graph_finalize(vdo_graph *g);

typedef struct vdo_lm_options {
  int max_iterations;       /* optimizer.optimize(N): 300 full batch, 100 partial (src/Optimizer.cc:1935, :807) */
  double gain_threshold;    /* SparseOptimizerTerminateAction::setGainThreshold; <= 0: action not installed */
  int max_trials;           /* maxTrialsAfterFailure, g2o default 10 */
  double pcg_rel_tol;       /* reduced-camera PCG: stop when sqrt(r.M^-1 r) <= tol * initial.  Default 1e-6: on BASELINE config 5 the LM run then
                               has the oracle's iteration count and ends within 9e-7 (poses) / 1.2e-6 m (points) of its direct-solve result (1e-8: 1e-8;
                               1e-5: 1.3e-5; the required agreement is 1e-4) -- measured table in DESIGN.md */
  int pcg_max_iterations;   /* default 2000 */
  int verbose;              /* per-iteration line on stderr, like optimizer.setVerbose(true) */
  int force_all_iterations; /* benchmarking: ignore every stop rule and run exactly max_iterations */
  double pcg_loose_tol;     /* forcing schedule of the inexact linear solves: while the previous LM iteration reduced chi2 by more than */
  double pcg_switch_gain;   /* pcg_switch_gain (relative), solve to pcg_loose_tol instead of pcg_rel_tol.  0 / 0: off (default) */
} vdo_lm_options;

typedef struct vdo_lm_stats {
  int iterations;           /* return value of SparseOptimizer::optimize */
  int trials;               /* total LM trials (linear solves) */
  int pcg_iterations;       /* total PCG iterations over all solves */
  double initial_chi2, final_chi2, final_lambda;
  double ms_linearize, ms_solve, ms_total; /* CUDA-event times on the context stream */
  int kernel_launches;      /* kernels launched by this optimize() call */
} vdo_lm_stats;

/* Converter (src/Converter.cc:25-41, 151-166) and the cv::Mat 4x4 product as the reference's float / double rounding rules (host-only):
 * toSE3Quat (rotation -> Eigen quaternion, w >= 0, normalised; q = x y z w), toCvMat (quaternion -> rotation, rounded to float),
 * toInvMatrix ([R^T | -R^T t], the translation accumulated in double and rounded once), A * B of two 4x4 CV_32F (float accumulation). */
int vdo_convert_to_se3quat(const float *T16, double *q4, double *t3);
int vdo_convert_to_cvmat(const double *q4, const double *t3, float *T16);
int vdo_convert_inv_matrix(const float *T16, float *out16);
int vdo_convert_mul4(const float *A16, const float *B16, float *out16);

/* sizeof() of a public struct as this library was built ("vdo_lm_options", "vdo_lm_stats", "vdo_tracker_params"; -1: unknown name): FFI
 * bindings that mirror the structs by hand (ctypes, cgo, JNI) check it at load time -- a binding that lags a struct extension would
 * otherwise have the library write past its buffer. */
int vdo_abi_struct_size(const char *name);

void vdo_lm_options_default(vdo_lm_options *o);

/* optimizer.optimize(max_iterations) (g2o/core/sparse_optimizer.cpp:354-427 with
 * OptimizationAlgorithmLevenberg::solve, g2o/core/optimization_algorithm_levenberg.cpp:61-164).
 * chi2_history (may be NULL): max_iterations+1 doubles, [0] = initial robust chi2. */
int vdo_graph_optimize(vdo_graph *g, const vdo_lm_options *opt, vdo_lm_stats *stats, double *chi2_history);

/* vertex->getEstimateData() (src/Optimizer.cc:2094-2172) */
int vdo_graph_get_vertices(const vdo_graph *g, double *se3, double *pt);
/* restore the estimates given to vdo_graph_set_vertices (device-to-device; used to repeat a solve) */
int vdo_graph_reset_vertices(vdo_graph *g);

/* sizes after finalize: out[0]=n_se3 out[1]=n_pt out[2]=n_pointxyz_edges out[3]=n_motion_edges out[4]=n_se3_edges
 * out[5]=n_prior out[6]=n_tracklets out[7]=device bytes held */
int vdo_graph_info(const vdo_graph *g, int64_t out[8]);
/* which solver paths the finalized graph uses: out[0]=tiled layout (0/1) out[1]=tiles out[2]=static tiles out[3]=width of the explicit
 * banded static block of the reduced matrix (0: matrix-free static product) out[4]=rows of that band out[5]=dense reduced-matrix path (0/1)
 * out[6]=preconditioner sharded by se3 path over the ranks (0/1) out[7]=se3 paths */
int vdo_graph_solver_info(const vdo_graph *g, int64_t out[8]);

/* Test hooks: one linearisation at the current estimates, returned in the caller's vertex numbering.
 * Hpp_diag: n_se3 x 36 (row-major 6x6 diagonal blocks), bp: n_se3 x 6, Hll_diag: n_pt (scalar: the 3x3
 * diagonal blocks are that scalar times I3 for scalar information), bl: n_pt x 3, chi2: robust chi2. */
int vdo_graph_debug_linearize(vdo_graph *g, double *Hpp_diag, double *bp, double *Hll_diag, double *bl, double *chi2);

/* ------------------------------------------------------------------------------------------------
 * .g2o files: the on-disk format of the graphs the reference dumps around every batch optimisation
 * (optimizer.save(...), src/Optimizer.cc:806,808,1934,1936 -> g2o/core/optimizable_graph.cpp:589-622, element syntax in
 * g2o/types/{vertex_se3,vertex_pointxyz,edge_se3,edge_se3_prior,edge_se3_pointxyz,types_dyn_slam3d,parameter_se3_offset}.cpp,
 * tags in g2o/types/types_slam3d.cpp:37-57).  Host-only.  Edge arrays use compact vertex indices (position of the vertex in
 * the file), the *_id arrays keep the file ids; information matrices are returned as written (upper triangle: 21 / 6
 * values).  Robust kernels are not part of the format, so vdo_graph_from_g2o takes the Huber deltas as arguments. */
typedef struct vdo_g2o vdo_g2o;
int vdo_g2o_read(const char *path, vdo_g2o **out);   /* on a parse error *out still carries the message (vdo_g2o_error) */
void vdo_g2o_free(vdo_g2o *g);
const char *vdo_g2o_error(const vdo_g2o *g);
/* out: n_se3, n_pt, n_prior, n_se3_edges, n_pointxyz_edges, n_motion_edges, n_fixed, n_offset_params */
int vdo_g2o_counts(const vdo_g2o *g, int64_t out[8]);
/* int arrays: se3_id pt_id fixed_id prior_v se3e_ij obs_cp ter_pph ; double arrays: se3 pt prior_Z prior_info se3e_Z
 * se3e_info obs_z obs_info ter_meas ter_info offset */
int vdo_g2o_get_i32(const vdo_g2o *g, const char *name, int *dst, int64_t cap);
int vdo_g2o_get_f64(const vdo_g2o *g, const char *name, double *dst, int64_t cap);
/* parsed file -> finalised graph; VDO_ERR_UNSUPPORTED unless every information matrix is w*I, motion measurements are
 * zero and the sensor offset is the identity, i.e. the family src/Optimizer.cc constructs */
int vdo_graph_from_g2o(vdo_ctx *ctx, const vdo_g2o *file, double delta_se3, double delta_pointxyz, double delta_motion, vdo_graph **out);
/* arrays in the layout of vdo_graph_add_* -> file; ids NULL: se3 vertex i -> i, point j -> n_se3 + j; precision <= 0: 17 digits */
int vdo_g2o_write(const char *path, int n_se3, const double *se3, const int *se3_id, int n_pt, const double *pt, const int *pt_id, int n_fixed,
                  const int *fixed_id, int n_prior, const int *prior_v, const double *prior_Z, const double *prior_w, int n_se3e, const int *se3e_ij,
                  const double *se3e_Z, const double *se3e_w, int n_obs, const int *obs_cp, const double *obs_z, const double *obs_w, int n_ter,
                  const int *ter_pph, const double *ter_w, int precision);

/* ------------------------------------------------------------------------------------------------
 * Per-frame input files of the reference's driver (example/vdo_slam.cc:98-141): PNG image / 16-bit disparity
 * (cv::imread UNCHANGED, :105-110), Middlebury .flo (cv::optflow::readOpticalFlow, :117), text label mask (LoadMask,
 * :253-450).  Host-only decoders; colour pixels in OpenCV order (BGR / BGRA), 16-bit samples host-endian. */
int vdo_io_png_info(const char *path, int *w, int *h, int *channels, int *bit_depth);
int vdo_io_read_png(const char *path, void *dst, size_t dst_bytes);            /* h x w x channels, uint8 or uint16 */
int vdo_io_read_png_gray_f32(const char *path, float *dst, int w, int h);      /* == imD.convertTo(imD_f, CV_32F) */
int vdo_io_flo_info(const char *path, int *w, int *h);
int vdo_io_read_flo(const char *path, float *dst, size_t dst_floats);          /* h x w x 2 (u, v) = CV_32FC2 */
int vdo_io_read_mask_txt(const char *path, int32_t *dst, int w, int h);        /* CV_32SC1, zeros where the file has zeros */

/* ------------------------------------------------------------------------------------------------
 * Result files and error metrics (the step after the path): System::SaveResults (src/System.cc:66-244) and
 * Tracking::GetMetricError (src/Tracking.cc:3243-3386), in the reference's float arithmetic and text format
 * (fixed, 9 decimals).  Per-frame entry lists are flattened: n_per_frame[i] entries for frame i (entry 0 = the camera,
 * skipped by both functions like the reference's `for j = 1`), labels / matrices of all frames back to back.  Host-only. */
int vdo_results_write_poses(const char *path, int start_frame, int n, const float *T16);   /* initial_/refined_stereo_new.txt, cam_pose_gt_stereo.txt */
/* obj_mot_stereo[_rf]_new.txt: body-frame motion toInvMatrix(pose_pre) * H * pose_pre ; pose_pre16 == NULL: as stored (obj_mot_gt.txt) */
int vdo_results_write_object_motions(const char *path, int start_frame, int n_frames, const int *n_per_frame, const int *labels, const float *H16,
                                     const float *pose_pre16);
int vdo_results_write_object_centres(const char *path, int start_frame, int n_frames, const int *n_per_frame, const int *labels, const float *centre3);
/* out4 = {camera t, camera R [deg], objects t, objects R [deg]} (means); each_obj_* have max_id - 1 entries (may be NULL) */
int vdo_metric_error(int n_cam, const float *cam16, const float *cam_gt16, int n_frames, const int *n_per_frame, const int *labels,
                     const unsigned char *obj_stat, const float *H16, const float *pose_pre16, const float *H_gt16, int max_id, float out4[4],
                     float *each_obj_t, float *each_obj_r, int *each_obj_count);

/* ------------------------------------------------------------------------------------------------
 * Per-frame joint optical-flow / SE(3) refinement.  Replaces Optimizer::PoseOptimizationFlow2 (object motion,
 * src/Optimizer.cc:2755-2972: prior information 0.5*I2, optimize(200)) and Optimizer::PoseOptimizationFlow2Cam (camera
 * pose, src/Optimizer.cc:2333-2542: prior 0.3*I2, optimize(100)), i.e. the g2o graph of one VertexSE3Expmap + n
 * VertexSBAFlow with EdgeSE3ProjectFlow2 (information 0.1*I2, Huber sqrt(0.04)) and EdgeFlowPrior edges, solved by
 * OptimizationAlgorithmLevenberg over BlockSolver_6_3 + LinearSolverDense.  The whole LM solve runs in one kernel.
 *
 *   mode       0 = camera (Flow2Cam), 1 = object (Flow2)
 *   quirk      1 = reproduce the arithmetic of 2-D flow vertices inside BlockSolver_6_3's 3x3 blocks (SURVEY.md H1;
 *              derived from source reading, the reference binary cannot be built here), 0 = intended 2x2 arithmetic
 *   pts        n x 2 f32  pixel of each point in the LAST frame   (pLastFrame->mvObjKeys / mvStatKeys[...].pt)
 *   depth      n     f32  its depth                               (mvObjDepth / mvStatDepth)
 *   flow       n x 2 f32  measured optical flow                   (mvObjFlowNext / mvFlowNext)
 *   K          4     f32  fx, fy, cx, cy                          (Frame::fx ...)
 *   Tcw_last   4x4   f32  row-major, pLastFrame->mTcw             (Twl is formed from it as the reference does, in float)
 *   T_init     4x4   f32  row-major, pCurFrame->mInitModel / mTcw
 * outputs
 *   T_out      4x4   f32  Converter::toCvMat(vSE3->estimate())
 *   flow_out   n x 2 f64  refined flow of every point (the caller adds it to the last-frame pixel for inliers)
 *   inlier     n     u8   1 if chi2 <= 0.04 (vIsOutlier[i] == false)
 *   stats      8     f64  [0] LM iterations (-1: n < 3, nothing optimised, T_out = identity) [1] trials [2] robust chi2
 *                         [3] lambda [4] inlier count
 * The batch form runs nprob independent problems (all objects of a frame) in one launch: offset has nprob+1 entries
 * into the concatenated pts / depth / flow / flow_out / inlier arrays; K, Tcw_last, T_init, T_out, stats are per problem. */
int vdo_pose_opt_flow2(vdo_ctx *ctx, int mode, int quirk, int n, const float *pts, const float *depth, const float *flow,
                       const float *K, const float *Tcw_last, const float *T_init, float *T_out, double *flow_out,
                       unsigned char *inlier, double *stats);
int vdo_pose_opt_flow2_batch(vdo_ctx *ctx, int quirk, int nprob, const int *mode, const int *offset, const float *pts,
                             const float *depth, const float *flow, const float *K, const float *Tcw_last,
                             const float *T_init, float *T_out, double *flow_out, unsigned char *inlier, double *stats);
/* measurement: re-run the last uploaded batch `reps` times on the device (no host copies), average ms per launch */
int vdo_pose_opt_flow2_time(vdo_ctx *ctx, int quirk, int nprob, int reps, float *ms_avg);

/* ------------------------------------------------------------------------------------------------
 * Image side of the per-frame path.  A vdo_frame keeps one frame's images resident in HBM: gray (u8), depth (f32),
 * optical flow (f32 x2, interleaved like CV_32FC2) and semantic mask (i32), all row-major width x height with no padding.
 * ------------------------------------------------------------------------------------------------ */
typedef struct vdo_frame vdo_frame;
int vdo_frame_create(vdo_ctx *ctx, int width, int height, vdo_frame **out);
void vdo_frame_destroy(vdo_frame *f);
/* H2D of the images TrackRGBD receives (include/System.h:49-51); any pointer may be NULL to keep what is resident */
int vdo_frame_upload(vdo_frame *f, const unsigned char *gray, const float *depth, const float *flow, const int *mask);
/* Tracking::GrabImageRGBD depth pre-processing (src/Tracking.cc:180-204): d < 0 -> 0, else bf / (d / factor), in place on the
 * resident depth; depth_out (may be NULL) receives the result so the caller's cv::Mat can be mutated like the reference does */
/* bf <= 0: clamp negatives to 0 only (the reference's VirtualKITTI branch) */
int vdo_frame_depth_prep(vdo_frame *f, float bf, float factor, float *depth_out);
/* ORBextractor::operator() (include/ORBextractor.h:47-49, src/ORBextractor.cc:1035-1110) on the resident gray image:
 * pyramid (cv::resize INTER_LINEAR chain), FAST-9/16 per 30-px cell with threshold fallback, octree distribution, IC_Angle.
 * Outputs are in the reference's keypoint order (level-major); max_out bounds the arrays; n_candidates (nlevels, may be NULL)
 * receives the per-level FAST candidate counts.  Descriptors are not produced (dead code in the reference, ORBextractor.cc:1091). */
int vdo_orb_extract(vdo_frame *f, int nfeatures, float scale_factor, int nlevels, int ini_th, int min_th, int max_out, float *x,
                    float *y, int *octave, float *response, float *angle, int *size, int *n_out, int *n_candidates);
/* Frame::Frame static candidates (src/Frame.cc:100-129, 181-194): keep ORB keypoints with mask == 0, 0 < depth <= th_depth,
 * non-zero flow whose target stays inside the image.  keep_idx = indices into the input, in order. */
int vdo_frame_filter_static(vdo_frame *f, int n, const float *kx, const float *ky, float th_depth, int *keep_idx, float *cx,
                            float *cy, float *fu, float *fv, float *depth, int *n_out);
/* Frame::SampleKeyPoints + Option II of Frame::Frame (src/Frame.cc:672-740, 130-194; UseSampleFeature: 1) on the resident images: the
 * VDO_SAMPLE_KEYPOINTS random pixels the reference draws from cv::RNG(seed) over a 20 x 20 grid (cell-major: cell i*20+j, column cell i,
 * row cell j; in draw order within a cell; duplicates kept), then the ones with mask == 0, 0 < depth <= th_depth, both flow components
 * non-zero and the flow target strictly inside the image (0 < x+fu < width, 0 < y+fv < height), in that order.  kx / ky: the kept pixels
 * (mvStatKeysTmp), cx / cy = x+fu / y+fv (mvCorres), fu / fv (mvFlowNext), depth (mvStatDepthTmp); max_out bounds these arrays.  seed 0
 * is cv::RNG(0), i.e. the stream of seed 0xffffffff.  raw_xy (may be NULL): the VDO_SAMPLE_KEYPOINTS x 2 unfiltered samples.
 * VDO_ERR_ARG when width or height is below 20 (the reference never leaves its sampling loop there). */
#define VDO_SAMPLE_KEYPOINTS 3000
int vdo_frame_sample_static(vdo_frame *f, uint32_t seed, float th_depth, int max_out, float *kx, float *ky, float *cx, float *cy, float *fu,
                            float *fv, float *depth, int *n_out, float *raw_xy);
/* Frame::Frame semi-dense object sampling (src/Frame.cc:200-228): raster scan with the given stride, mask != 0,
 * 0 < depth < th_depth_obj, flow target inside the image; outputs in raster (push_back) order */
int vdo_frame_sample_objects(vdo_frame *f, float th_depth_obj, int step, int max_out, int *x, int *y, float *cx, float *cy,
                             float *fx, float *fy, float *depth, int *label, int *n_out);
/* Tracking::GetSceneFlowObj with Frame::UnprojectStereoObject (src/Tracking.cc:1278-1364, src/Frame.cc:521-555):
 * flow3d[i] = X_w(cur, i) - X_w(prev, i) in float; valid[i] = both labels > 0 (otherwise the reference sets vObjLabel = -1).
 * Tcw_* are 4x4 row-major f32 (Frame::mTcw); Xw_prev (n x 3, may be NULL) returns the previous-frame world points. */
int vdo_scene_flow(vdo_ctx *ctx, int n, const float *u_prev, const float *v_prev, const float *z_prev, const float *Tcw_prev,
                   const float *u_cur, const float *v_cur, const float *z_cur, const float *Tcw_cur, const float *K,
                   const int *label_prev, const int *label_cur, float *flow3d, float *Xw_prev, unsigned char *valid);
/* 7x7 sigma-2 Gaussian blur of every pyramid level + rotated-BRIEF descriptors (src/ORBextractor.cc:1083-1084, 97-136, pattern :139-397) of the
 * keypoints of the last vdo_orb_extract call (which must have returned angles).  The reference allocates the descriptor matrix and never fills
 * it (the computeDescriptors call is commented out, :1091); this is that call.  desc_out: n x 32 bytes in vdo_orb_extract's keypoint order. */
int vdo_orb_describe(vdo_frame *f, int n, unsigned char *desc_out);
int vdo_frame_debug_blur(vdo_frame *f, int level, unsigned char *img_out);   /* test hook: blurred level of the last vdo_orb_describe */
/* test hook: pyramid level and FAST score map (u8, cv::cornerScore clipped at 0) of the last vdo_orb_extract call */
int vdo_frame_debug_level(vdo_frame *f, int level, unsigned char *img_out, unsigned char *score_out, int *w_out, int *h_out);
/* measurement: device time of the ORB front end (pyramid + FAST score maps) on the resident image */
int vdo_orb_time(vdo_frame *f, int reps, float *ms_avg);

/* ---- initial model (SURVEY.md 8 row A10 / next-row N1) ------------------------------------------------------------------
 * vdo_init_model_batch  <- Tracking::GetInitModelCam / GetInitModelObj (src/Tracking.cc:1614-1715, 1717-1849), including the
 *   cv::solvePnPRansac(pre_3d, cur_2d, K, 0, rvec, tvec, false, iters=500, thr=0.4, conf=0.98, inliers, SOLVEPNP_AP3P) call
 *   (OpenCV 3.4; engine restated in oracle/pnp_ransac.c).  One problem per camera / object: points offsets[p]..offsets[p+1] of
 *   obj3d (pre_3d, n x 3 f32, world) and img2d (cur_2d, n x 2 f32).  K4 = fx, fy, cx, cy (Frame::fx.. / mK).  T_mm (nprob x 16,
 *   4x4 row-major f32) is the constant-motion model (mVelocity*mLastFrame.mTcw, or mTcw*vObjMod[PreObjID]); has_mm[p] = 0 for an
 *   object with no previous motion (PreObjID == -1).  Outputs: T_init (nprob x 16: `output`), n_sub[p] and sub_idx (the chosen
 *   inlier subset as ascending LOCAL indices, stored from offsets[p]); info (nprob x 8 ints: inliers.rows, MM_inlier.size(),
 *   motion model used, n_sub, RANSAC iterations run, winning iteration, valid minimal solves, 0); Rt_refit / Rt_hyp
 *   (nprob x 12 f64 [R row-major | t], may be NULL): refitted model and winning hypothesis (test hooks). */
int vdo_init_model_batch(vdo_ctx *ctx, int nprob, const int *offsets, const float *obj3d, const float *img2d, const float *K4, int iters,
                         double thr, double conf, const float *T_mm, const unsigned char *has_mm, float *T_init, int *n_sub, int *sub_idx,
                         int *info, double *Rt_refit, double *Rt_hyp);
/* kernels launched so far by vdo_init_model_batch on this context (bench accounting) */
int vdo_init_model_launches(vdo_ctx *ctx);

/* ---- tracking bookkeeping (SURVEY.md 8 rows A13, A15, A16) -----------------------------------------------------------
 * vdo_tracklets_build  <- Tracking::GetStaticTrack / GetDynamicTrackNew (src/Tracking.cc:2201-2307, 2309-2421).
 *   Row i (0-based, i = frame pair id) holds row_begin[i+1]-row_begin[i] features of frame i+1; assoc[k] is the index of the
 *   same feature in frame i's row (Map::vnAssoSta / vnAssoDyn), -1 = no correspondence; labels (NULL for the static map) is
 *   Map::vnFeatLabel (the dynamic-object id of the feature).  Tracklets come out in the reference's creation order as CSR:
 *   entry e of tracklet t is (trk_frame[e], trk_feat[e]) = TrackLets[t][.] = (frame id, feature id); obj_id[t] = ObjLab[t].
 *   Host-only (no device work).  Returns VDO_ERR_ARG (with *n_trk set) when max_tracklets / max_entries are too small. */
int vdo_tracklets_build(int n_rows, const int *row_begin, const int *assoc, const int *labels, int max_tracklets, int max_entries,
                        int *n_trk, int *trk_begin, int *trk_frame, int *trk_feat, int *obj_id);
/* vdo_update_mask  <- Tracking::UpdateMask (src/Tracking.cc:2997-3110).  cur / last are resident frames (mask of both, flow of
 *   last).  sem_label_last / corres_x / corres_y are the last frame's vSemObjLabel and mvObjCorres (n object points).  The
 *   current mask is updated in place on the device; mask_out (h*w int, may be NULL) receives it (the caller's mSegMap);
 *   warped_labels (may be NULL, sized for the number of distinct labels) lists the objects whose mask was recovered. */
int vdo_update_mask(vdo_frame *cur, vdo_frame *last, int n, const int *sem_label_last, const float *corres_x, const float *corres_y,
                    int *mask_out, int *n_warped, int *warped_labels);
/* vdo_dyn_obj_tracking  <- Tracking::DynObjTracking (src/Tracking.cc:1366-1612; ground-truth bookkeeping :1531-1544 excluded).
 *   n object points of the current frame: sem_label (vSemObjLabel), obj_label (vObjLabel, in/out), kx/ky (mvObjKeys),
 *   depth (mvObjDepth), flow3d (vFlow_3d, n x 3), sem_label_last (mLastFrame.vSemObjLabel); the last frame's object table
 *   (nSemPosition, bObjStat, nModLabel); rows/cols of the image, shrink_row/col (25/50 for KITTI, 0 otherwise),
 *   sf_mg_thres / sf_ds_thres / th_depth_obj (fSFMgThres, fSFDsThres, mThDepthObj), f_id and max_id (in/out).
 *   Outputs: the kept objects as CSR over point indices (return value ObjIdNew), mod_label (nModLabel), sem_position
 *   (nSemPosition). */
int vdo_dyn_obj_tracking(vdo_ctx *ctx, int n, const int *sem_label, int *obj_label, const float *kx, const float *ky, const float *depth,
                         const float *flow3d, const int *sem_label_last, int n_last_obj, const int *last_sem_position,
                         const unsigned char *last_obj_stat, const int *last_mod_label, int rows, int cols, int shrink_row, int shrink_col,
                         float sf_mg_thres, float sf_ds_thres, float th_depth_obj, int f_id, int *max_id, int max_objects,
                         int *n_objects, int *obj_begin, int *obj_idx, int *mod_label, int *sem_position);

/* vdo_renew_frame_info  <- Tracking::RenewFrameInfo (src/Tracking.cc:2660-2995).  `cur` holds the current images (prepared depth,
 *   updated mask, flow).  Static part: tm_sta (TM_sta = TemperalMatch_subset after Flow2Cam, -1 = outlier) indexes stat_keys
 *   (mCurrentFrame.mvStatKeys, n_stat x 2); samp_keys (n_samp x 2) is mvKeys (ORB) or mvStatKeysTmp (nUseSampleFea == 1);
 *   max_num_sta = nMaxTrackPointBG.  Object part: inl_begin / inl_idx = vnObjInlierID (CSR over n_obj objects), obj_stat =
 *   bObjStat, sem_position = nSemPosition, mod_label = nModLabel, obj_keys / obj_label = mvObjKeys / vObjLabel (n_objkeys),
 *   tmp_* = this frame's fresh semi-dense samples (mvTmpObjKeys, mvTmpObjDepth, mvTmpSemObjLabel, mvTmpObjFlowNext, mvTmpObjCorres;
 *   n_tmp), max_num_obj = nMaxTrackPointOBJ.  K4 = fx, fy, cx, cy; Twc = Converter::toInvMatrix(mTcw), 4x4 row-major f32.
 *   Outputs (caller-allocated, capacities cap_sta / cap_obj): static mvStatKeysTmp, mvCorres, mvFlowNext, nStaInlierID,
 *   mvStatDepthTmp, mvStat3DPointTmp; objects mvObjKeys, mvObjDepth, mvObjCorres, mvObjFlowNext, vSemObjLabel, nDynInlierID,
 *   vObjLabel, mvObj3DPoint.  The depth limits 40 / 25 are hard-coded like in the reference (:2691, :2849). */
int vdo_renew_frame_info(vdo_frame *cur, int n_tm, const int *tm_sta, int n_stat, const float *stat_keys, int n_samp, const float *samp_keys,
                         int max_num_sta, int n_obj, const int *inl_begin, const int *inl_idx, const unsigned char *obj_stat,
                         const int *sem_position, const int *mod_label, int n_objkeys, const float *obj_keys, const int *obj_label, int n_tmp,
                         const float *tmp_keys, const float *tmp_depth, const int *tmp_sem, const float *tmp_flow, const float *tmp_corres,
                         int max_num_obj, const float *K4, const float *Twc, int cap_sta, int *n_sta_out, float *sta_keys, float *sta_corres,
                         float *sta_flow, int *sta_inlier_id, float *sta_depth, float *sta_3d, int cap_obj, int *n_obj_out, float *o_keys,
                         float *o_depth, float *o_corres, float *o_flow, int *o_sem, int *o_inlier_id, int *o_label, float *o_3d);

/* depth and mask label at the truncated pixel of each key (x, y interleaved, n x 2 f32); 0 / 0 outside the image.  The
 * "update current frame from last" look-ups of Tracking::GrabImageRGBD (src/Tracking.cc:262-312). */
int vdo_frame_gather(vdo_frame *f, int n, const float *keys, float *depth_out, int *mask_out);
int vdo_frame_read_mask(vdo_frame *f, int *mask_out);   /* D2H of the resident (possibly updated) semantic mask */

/* ------------------------------------------------------------------------------------------------
 * Whole per-frame path: System::TrackRGBD -> Tracking::GrabImageRGBD -> Tracking::Track (include/System.h:49-51,
 * src/Tracking.cc:164-648, 650-1212) sequenced over the stages above, with the per-frame state of `Frame` and the slice of `Map`
 * the batch optimisers read kept inside the tracker.  Settings mirror the YAML keys Tracking::Tracking reads
 * (src/Tracking.cc:57-162; defaults = example/kitti-0000-0013.yaml).
 * ------------------------------------------------------------------------------------------------ */
typedef struct vdo_tracker vdo_tracker;
typedef struct vdo_tracker_params {
  int width, height;                 /* Camera.width / Camera.height */
  float fx, fy, cx, cy;              /* Camera.fx .. */
  float bf, depth_factor;            /* Camera.bf, DepthMapFactor */
  float th_depth_bg, th_depth_obj;   /* ThDepthBG, ThDepthOBJ */
  int max_track_bg, max_track_obj;   /* MaxTrackPointBG, MaxTrackPointOBJ */
  float sf_mg_thres, sf_ds_thres;    /* SFMgThres, SFDsThres */
  int n_features; float scale_factor; int n_levels, ini_th_fast, min_th_fast;   /* ORBextractor.* */
  int is_kitti;                      /* mTestData == KITTI: boundary shrink 25 / 50 px (src/Tracking.cc:1405-1409) */
  int quirk;                         /* see vdo_pose_opt_flow2 */
  int window_size, overlap_size;     /* WINDOW_SIZE, OVERLAP_SIZE */
  int local_batch;                   /* bLocalBatch: run PartialBatchOptimization inside vdo_tracker_track on the reference's schedule
                                        ((f_id - OVERLAP + 1) % (WINDOW - OVERLAP) == 0 && f_id >= WINDOW - 1, src/Tracking.cc:1150-1160) */
  int dataset;                       /* ChooseData / mTestData (src/Tracking.cc:150-160): 1 OMD, 2 KITTI, 3 VirtualKITTI; 0 = KITTI when is_kitti else OMD.
                                        OMD and KITTI convert the raw disparity to depth (bf / (d / factor)); VirtualKITTI only clamps negatives
                                        to 0 (src/Tracking.cc:180-204) */
  int use_sample_feature;            /* UseSampleFeature: 1 = background keypoints from vdo_frame_sample_static instead of the ORB keypoints
                                        (ORB still runs: a frame without ORB keypoints stays empty, src/Frame.cc:97-98), and the RenewFrameInfo
                                        top-up draws from that filtered sample list (src/Tracking.cc:2718-2721) */
  unsigned sample_seed;              /* 0: every frame seeds with (unsigned)time(NULL) read when it is built, like src/Frame.cc:674; otherwise every
                                        frame uses this seed (what the reference does for frames built within the same second).  The seed of the
                                        last frame is vdo_tracker_get("sample_seed") */
} vdo_tracker_params;
void vdo_tracker_params_default(vdo_tracker_params *p);
int vdo_tracker_create(vdo_ctx *ctx, const vdo_tracker_params *params, vdo_tracker **out);
void vdo_tracker_destroy(vdo_tracker *t);
const char *vdo_tracker_last_error(const vdo_tracker *t);
/* One frame.  gray: h x w u8; depth: h x w f32 raw disparity*factor as example/vdo_slam.cc passes it -- when writeback != 0 it is
 * overwritten with metric depth like the reference does to the caller's cv::Mat (src/Tracking.cc:180-204); flow: h x w x 2 f32;
 * mask: h x w i32 -- when writeback != 0 it receives the propagated labels (UpdateMask, :3062).  gt_sem_ids: semantic ids that have a
 * ground-truth object pose in this frame (vObjPose_gt[i][1]); the reference only estimates motion for objects present in the
 * ground truth of both frames (:767-810).  Tcw_out: 4x4 row-major f32 = the returned mCurrentFrame.mTcw.
 * width / height: size of the four buffers; VDO_ERR_ARG unless they equal the tracker's (the buffers are read -- and with writeback
 * written -- as width x height arrays). */
int vdo_tracker_track(vdo_tracker *t, int width, int height, const unsigned char *gray, float *depth, const float *flow, int *mask, int n_gt,
                      const int *gt_sem_ids, int writeback, float *Tcw_out);
/* Named read-back of the frame state after the last call ('f' arrays are f32, the others i32; out may be NULL to query the size):
 * Tcw mVelocity mvKeys mvStatKeysTmp mvStatDepthTmp mvCorres mvFlowNext mvStat3DPointTmp nStaInlierID mvObjKeys mvObjDepth
 * mvObjCorres mvObjFlowNext mvObj3DPoint vSemObjLabel vObjLabel nDynInlierID vFlow_3d nModLabel nSemPosition bObjStat vObjMod
 * vObjCentre3D TemperalMatch_subset max_id f_id; stage_ms (9 x f32, accumulated host wall-clock per stage since creation: upload+depth, mask,
 * frame build (ORB + static filter + object samples), look-ups, initial camera model, camera LM, objects, renewal, windowed BA);
 * local_ba (2 x i32: windowed optimisations run, their LM iterations); sample_seed (1 x u32: the seed the last frame sampled with, 0 when it did
 * not sample) */
int vdo_tracker_get(const vdo_tracker *t, const char *name, void *out, int cap_elems, int *n_elems);

/* Map -> factor graph -> optimise -> write back (SURVEY.md 8f N2): mode 0 = Optimizer::PartialBatchOptimization(pMap, K, WINDOW_SIZE)
 * (src/Optimizer.cc:42-1230) over the last window_size frames, mode 1 = Optimizer::FullBatchOptimization(pMap, K) (:1232-2175),
 * on the map the tracker accumulated (Tracking.cc:1016-1070).  opt may be NULL (the reference's optimize(100 | 300) and gain
 * thresholds 1e-3 | 1e-4).  info (may be NULL, 6 ints): vertices se3 / point, edges prior / se3 / point-observation / landmark-motion. */
int vdo_tracker_batch_optimize(vdo_tracker *t, int mode, const vdo_lm_options *opt, vdo_lm_stats *stats, int *info);
/* test hook: the arrays the builder passes to vdo_graph_* for a mode.  f64 names: se3 pt prior_Z prior_w se3e_Z se3e_w se3e_delta
 * obs_z obs_w obs_delta ter_w ter_delta; i32 names: prior_v se3e_ij obs_cp ter_pph.  out may be NULL to query the element count. */
int vdo_tracker_graph_export(vdo_tracker *t, int mode, const char *name, void *out, int cap_elems, int *n_elems);
/* map read-back (include/Map.h:34-84): vmCameraPose / vmCameraPose_RF (n_frames x 16 f32: the windowed BA refines the first, the full
 * batch the second, src/Optimizer.cc:1058-1101 / :2094-2133), vmRigidMotion / vmRigidMotion_RF (every frame's motions concatenated, 16 f32
 * each, entry 0 = camera motion), vmRigidCentre (3 f32 each, same order), vnRMLabel (i32, same order), n_per_frame (entries per frame,
 * i32), n_frames (i32) */
int vdo_tracker_map_get(const vdo_tracker *t, const char *name, void *out, int cap_elems, int *n_elems);
/* Externally built maps -- the input of Optimizer::FullBatchOptimization(Map*, K) / PartialBatchOptimization(Map*, K, WINDOW_SIZE)
 * (include/Optimizer.h:29-30): create a handle with params.width == params.height == 0 (intrinsics, window_size and overlap_size are used),
 * push the Map frame by frame, run vdo_tracker_batch_optimize and read vmCameraPose[_RF] / vmRigidMotion[_RF] / vp3DPointSta / vp3DPointDyn
 * (xyz per feature, all frames concatenated) back with vdo_tracker_map_get.  Frame 0: n_mot = 0, asso / label arrays ignored. */
int vdo_tracker_map_push(vdo_tracker *t, int n_sta, const float *feat_sta, const float *dep_sta, const float *p3d_sta, const int *asso_sta, int n_dyn,
                         const float *feat_dyn, const float *dep_dyn, const float *p3d_dyn, const int *asso_dyn, const int *feat_label,
                         const float *camera_pose16, int n_mot, const float *rigid_motion16, const int *rm_label);

/* Measurement hook (bench.py roofline): runs one kernel (or kernel group) of the batch path `reps` times back to back
 * on the context stream between two CUDA events, after one untimed warm-up launch, and returns the average in ms.
 * The graph must have been optimised at least once (buffers hold a valid linearisation / factorisation).
 * names: "lin_tracklets" "chi2_tracklets" "lin_vertex_obs" "lin_vertex_ter" "lin_se3_edges" "linearize" (all four)
 *        "factor_landmarks" "precond" (assembly + PCR factorisation) "schur_landmarks" "schur_vertex_obs"
 *        "schur_vertex_ter" "hpp_mul" "pcg_dot" "pcg_step" "pcg_iterate8" (8 PCG iterations as launched in a solve)
 *        "schur_static" "schur_chains" "lin_static" "lin_chains" (the two halves of the landmark passes) "pcg_step_a" */
int vdo_graph_time_kernel(vdo_graph *g, const char *name, int reps, float *ms_avg);

#ifdef __cplusplus
}
#endif
#endif
