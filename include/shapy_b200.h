/* shapy_b200 -- C ABI of the B200-native SHAPY inference hot path.
 *
 * Every entry point is `extern "C"`, takes plain pointers / sizes / a CUDA stream
 * (passed as void* so the header needs no CUDA include) and returns 0 on success or
 * a negative shapy_b200 error / positive cudaError_t code; shapy_last_error() gives
 * the message.  No torch types.  All device work is stream-ordered on `stream`; no
 * call synchronises the device.  Outputs are caller-owned device buffers.
 *
 * What each entry point replaces in the reference (paths relative to the reference
 * repo, see SURVEY.md section 8):
 *
 *   shapy_smplx_*        lbs()                      regressor/human_shape/models/body_models/lbs.py:99-196
 *                        SMPLX.forward              regressor/human_shape/models/body_models/body_models.py:628-767
 *                        SMPL.forward_shape         body_models.py:292-302
 *                        ContinuousRotReprDecoder   regressor/human_shape/models/common/pose_utils.py:138-153
 *                        WeakPerspectiveCamera      regressor/human_shape/models/camera/camera_projection.py:181-213
 *   shapy_measure_*      BodyMeasurements.forward   mesh-mesh-intersection/body_measurements/body_measurements.py:217-246
 *   shapy_mmi_forward    mesh_to_mesh_forward       mesh-mesh-intersection/src/mesh_mesh_intersect.cpp:36-64
 *                                                   + src/mesh_mesh_intersect_cuda_op.cu:969-1079
 *   shapy_head_*         IterativeRegression.forward regressor/human_shape/models/common/networks.py:536-592
 *   shapy_hrnet_*        HighResolutionNet.forward  regressor/human_shape/models/backbone/hrnet.py:426-498
 */
#ifndef SHAPY_B200_H_
#define SHAPY_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SHAPY_OK 0
#define SHAPY_ERR_ARG (-1)      /* bad argument (null pointer, unsupported size) */
#define SHAPY_ERR_STATE (-2)    /* object not bound / wrong device */
#define SHAPY_ERR_UNSUPPORTED (-3)
#define SHAPY_ERR_OVERFLOW (-4) /* a fixed-capacity device buffer overflowed */

const char *shapy_last_error(void);
int shapy_version(void);
/* number of kernels this library launched since process start (all entry points) */
long long shapy_launch_count(void);

/* ------------------------------------------------------------------ SMPL-X */
typedef struct shapy_smplx shapy_smplx_t;

/* Dense model tensors exactly as the reference registers them as buffers
 * (body_models.py:112-166, 563-597).  HOST pointers, fp32 / int64, row-major. */
typedef struct {
  int num_verts;               /* V  (10475) */
  int num_joints;              /* J  (55)    */
  int num_betas;               /* NB (10)  shapedirs is (V,3,NB) */
  int num_expr;                /* NE (10)  expr_dirs is (V,3,NE); may be 0 */
  int num_faces;               /* F  (20908) */
  const float *v_template;     /* (V,3) */
  const float *shapedirs;      /* (V,3,NB) */
  const float *expr_dirs;      /* (V,3,NE) or NULL */
  const float *posedirs;       /* ((J-1)*9, V*3) */
  const float *J_regressor;    /* (J,V) */
  const float *lbs_weights;    /* (V,J) */
  const int64_t *parents;      /* (J), parents[0] = -1 */
  const int64_t *faces;        /* (F,3) */
  int num_static_lmk;          /* 51 */
  const int64_t *lmk_faces_idx;        /* (L) */
  const float *lmk_bary_coords;        /* (L,3) */
  int num_dyn_lmk;             /* 17, 0 disables use_face_contour */
  int num_dyn_rows;            /* 79 */
  const int64_t *dynamic_lmk_faces_idx;   /* (rows, D) */
  const float *dynamic_lmk_bary_coords;   /* (rows, D, 3) */
  int neck_chain_len;          /* 6 */
  const int64_t *neck_kin_chain;       /* e.g. [15,12,9,6,3,0] */
  int num_extra;               /* 14 rows of the J14 regressor, 0 disables */
  const float *extra_joint_regressor;  /* (num_extra, V) */
  int num_overwrite;           /* len(source_idxs) */
  const int64_t *source_idxs;  /* joints[:, source] = reg[:, target] */
  const int64_t *target_idxs;
} shapy_smplx_desc_t;

int shapy_smplx_create(shapy_smplx_t **out, const shapy_smplx_desc_t *desc);
void shapy_smplx_destroy(shapy_smplx_t *m);
int shapy_smplx_num_keypoints(const shapy_smplx_t *m);          /* J + L + D (123) */
const int32_t *shapy_smplx_faces_i32(const shapy_smplx_t *m);   /* device (F,3) int32 */
size_t shapy_smplx_workspace_bytes(const shapy_smplx_t *m, int batch);

/* 6D -> rotation matrices: raw (n, 6) row-major 3x2 -> rot (n, 3, 3). */
int shapy_decode_rot6d(const float *raw, int n, float *rot, void *stream);

/* Full SMPL-X evaluation for `batch` bodies.
 *   betas   (B, NB)                 device fp32
 *   rot     (B, n_rot, 3, 3)        rotations of the first n_rot joints of the full pose
 *                                   [global, body(21), jaw, leye, reye, lhand(15), rhand(15)];
 *                                   the remaining joints are identity (SHAPY_A: n_rot = 22)
 *   expr    (B, NE) or NULL (zeros)
 *   camera  (B, 3) or NULL; when given, proj_joints = softplus(c0) * (joints_xy + c[1:3])
 * outputs (any may be NULL): vertices (B,V,3), v_shaped (B,V,3), joints (B,K,3), proj_joints (B,K,2)
 */
int shapy_smplx_forward(const shapy_smplx_t *m, const float *betas, const float *rot, int n_rot,
                        const float *expr, const float *camera, int batch, float *vertices, float *v_shaped,
                        float *joints, float *proj_joints, void *workspace, size_t workspace_bytes,
                        void *stream);

/* v_shaped = v_template + shapedirs . betas  (T-pose path, BASELINE configs 1 and 4) */
int shapy_smplx_forward_shape(const shapy_smplx_t *m, const float *betas, int batch, float *v_shaped,
                              void *stream);

/* Backward of shapy_smplx_forward_shape: grad_betas (B, num_betas) = shapedirs^T . grad_v_shaped (B,V,3), summed in a
 * fixed order (a body's result does not depend on its position in the batch). */
int shapy_smplx_shape_backward(const shapy_smplx_t *m, const float *grad_v_shaped, int batch, float *grad_betas,
                               void *stream);

/* ------------------------------------------------------- virtual measurements */
typedef struct {
  int face_idx[5];      /* head_top, left_heel, chest, waist, hips landmark faces */
  float bc[5][3];       /* barycentrics */
} shapy_measure_landmarks_t;

/* v_shaped (B,V,3), faces int32 (F,3) device.  out (B,5) = mass, height, chest, waist, hips.
 * plane_points (optional, (B,3,max_points,3)) / plane_counts (optional, (B,3) int32) receive the
 * reference-selected intersection points of each slicing plane.  status (device int32[1], may be
 * NULL) is set non-zero if any plane exceeded max_points (SHAPY_ERR_OVERFLOW semantics). */
int shapy_measure_forward(const float *v_shaped, const int32_t *faces, int batch, int num_verts, int num_faces,
                          const shapy_measure_landmarks_t *lm, float *out, float *plane_points,
                          int32_t *plane_counts, int max_points, int32_t *status, void *stream);

/* Same on explicit triangles (B,F,3,3) -- the tensor BodyMeasurements.forward receives. */
int shapy_measure_forward_tris(const float *triangles, int batch, int num_faces,
                               const shapy_measure_landmarks_t *lm, float *out, float *plane_points,
                               int32_t *plane_counts, int max_points, int32_t *status, void *stream);

/* Backward of shapy_measure_forward: grad_out (B,5) -> grad_v (B,V,3), the first derivative of
 * sum_j grad_out[b][j] * out[b][j] with the intersection barycentrics and the slicing heights held constant (the
 * reference computes them under no_grad).  Recomputes the forward's point sets and hulls; no float atomics, so the
 * result is bit-reproducible.  A NaN circumference with a non-zero grad_out entry makes that body's gradient NaN; a
 * zero entry contributes nothing.  workspace: shapy_measure_backward_workspace_bytes(num_verts, num_faces) bytes
 * (the vertex -> face adjacency, rebuilt by every call).  num_verts is limited by the shared-memory staging
 * (SMPL-X and SMPL fit); beyond it the call fails with SHAPY_ERR_ARG. */
size_t shapy_measure_backward_workspace_bytes(int num_verts, int num_faces);
int shapy_measure_backward(const float *v_shaped, const int32_t *faces, int batch, int num_verts, int num_faces,
                           const shapy_measure_landmarks_t *lm, const float *grad_out, float *grad_v,
                           void *workspace, size_t workspace_bytes, void *stream);

/* Same on explicit triangles: grad_tris (B,F,3,3), mirroring shapy_measure_forward_tris (and its capacities). */
int shapy_measure_backward_tris(const float *triangles, int batch, int num_faces,
                                const shapy_measure_landmarks_t *lm, const float *grad_out, float *grad_tris,
                                void *stream);

/* Drop-in for mesh_mesh_intersect_cuda.mesh_to_mesh_forward: query (B,Q,3,3), target (B,F,3,3) fp32;
 * collision_faces (B,Q*M) int64 pre-filled by the callee with -1; collision_bcs (B,Q*M,2,3) with 0. */
size_t shapy_mmi_workspace_bytes(int batch, int num_query, int num_target);
int shapy_mmi_forward(const float *query, const float *target, int batch, int num_query, int num_target,
                      int max_collisions, int64_t *collision_faces, float *collision_bcs, void *workspace,
                      size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------ regression head */
/* params_out (num_stages, B, P).  W0 (H0, F+P), W1 (H1, H0), W2 (P, H1) row-major as nn.Linear stores
 * them; mean (P).  workspace >= shapy_head_workspace_bytes. */
size_t shapy_head_workspace_bytes(int batch, int feat_dim, int param_dim, int h0, int h1);
int shapy_head_forward(const float *feats, int batch, int feat_dim, int param_dim, int h0, int h1,
                       const float *W0, const float *b0, const float *W1, const float *b1, const float *W2,
                       const float *b2, const float *mean, int num_stages, float *params_out, void *workspace,
                       size_t workspace_bytes, void *stream);

/* The MLP has no activation, so a stage collapses exactly (in real arithmetic) to p' = p + Mf f + Mp p + c.
 * MfT (F, P) = (W2 W1 W0[:, :F])^T, MpT (P, P) = (W2 W1 W0[:, F:])^T, c (P) = W2 (W1 b0 + b1) + b2, contracted by
 * the caller in fp64.  workspace >= B * P * 4 bytes. */
int shapy_head_forward_collapsed(const float *feats, int batch, int feat_dim, int param_dim, const float *MfT,
                                 const float *MpT, const float *c, const float *mean, int num_stages,
                                 float *params_out, void *workspace, size_t workspace_bytes, void *stream);

/* -------------------------------------------------------------------- HRNet */
typedef struct shapy_hrnet shapy_hrnet_t;

/* One convolution of the backbone, BN already folded by the caller's choice: the library folds
 * scale into the weights itself when `bn_*` are given.  HOST pointers. */
typedef struct {
  int cin, cout, ksize, stride; /* ksize 1 or 3, stride 1 or 2, padding ksize/2 */
  const float *weight;          /* (cout, cin, k, k) */
  const float *bias;            /* (cout) or NULL */
  const float *bn_weight, *bn_bias, *bn_mean, *bn_var; /* (cout) each or all NULL */
  float bn_eps;
} shapy_conv_desc_t;

enum { SHAPY_OP_STEM = 0, SHAPY_OP_CONV = 1, SHAPY_OP_FUSE = 2, SHAPY_OP_POOL = 3 };

/* Program of the network: a flat list of ops over numbered activation slots.  A slot is a
 * (B, H/div, W/div, C) NHWC tensor; outputs may write a channel slice of a wider slot
 * (out_coff / slot channels) which is how the 4x384 concat is formed without a copy. */
typedef struct {
  int kind;          /* SHAPY_OP_* */
  int conv;          /* index into the conv table (STEM / CONV) */
  int in_slot;       /* -1 = network input (STEM) */
  int out_slot, out_coff;
  int res_slot;      /* residual added before ReLU, -1 none */
  int relu;
  /* FUSE: out = relu(sum_i up(in_i)); in_i at scale 2^shift_i coarser than out (nearest) */
  int n_in;
  int fuse_in[4];
  int fuse_shift[4];
  /* Execution lane (0..SHAPY_MAX_LANES-1).  Ops of one lane run in program order on one CUDA stream; ops of
   * different lanes may run concurrently (the independent branches of a HighResolutionModule, reference
   * hrnet.py:175-193).  The executor derives every cross-lane ordering itself from the slots an op reads and
   * writes (RAW, WAR and WAW), so the lane is a scheduling hint only: any assignment gives the serial result. */
  int lane;
} shapy_op_t;
enum { SHAPY_MAX_LANES = 4 };

typedef struct {
  int channels;      /* total channels of the slot */
  int div;           /* spatial divisor w.r.t. the network input (4, 8, 16, 32, 2) */
} shapy_slot_t;

/* mode: 0 = fp16 operands, single pass (BASELINE config 2);
 *       1 = split-fp16 (hi + lo planes, 3 MMAs per tile, ~fp32 accuracy; parity mode);
 * engine: 0 = tcgen05 implicit GEMM where the shape allows, 1 = SIMT fp32 everywhere (debug). */
int shapy_hrnet_create(shapy_hrnet_t **out, const shapy_conv_desc_t *convs, int n_convs, const shapy_op_t *ops,
                       int n_ops, const shapy_slot_t *slots, int n_slots, int feat_slot, int mode, int engine);
void shapy_hrnet_destroy(shapy_hrnet_t *p);
size_t shapy_hrnet_workspace_bytes(const shapy_hrnet_t *p, int batch, int height, int width);
/* images (B,3,H,W) fp32 NCHW device; feats (B, C_feat) fp32 device. */
int shapy_hrnet_forward(shapy_hrnet_t *p, const float *images, int batch, int height, int width, float *feats,
                        void *workspace, size_t workspace_bytes, void *stream);
/* copies slot `slot` (after a forward) to dst as fp32 NCHW (B,C,H/div,W/div); for tests. */
int shapy_hrnet_read_slot(shapy_hrnet_t *p, int slot, float *dst, void *stream);
double shapy_hrnet_flops(const shapy_hrnet_t *p, int batch, int height, int width);

/* Standalone conv for unit tests of the implicit-GEMM kernel: x (B,H,W,Cin) fp32 NHWC device,
 * y (B,Ho,Wo,Cout) fp32 NHWC device, res optional (same shape as y). */
int shapy_conv_test(const shapy_conv_desc_t *conv, const float *x, const float *res, int batch, int height,
                    int width, int relu, int mode, int engine, float *y, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Input stage (SURVEY.md 8f rank 1): uint8 full images + crop windows -> normalised fp32 NCHW crops.
 * Replaces, per detected person, the reference's CPU chain
 *   read_img        regressor/human_shape/utils/img_utils.py:57-61         (uint8 -> float32 / 255, clip)
 *   crop            regressor/human_shape/utils/transf_utils.py:51-96      (window [ul, br), zero padding,
 *                                                                           cv2.resize INTER_LINEAR to size x size)
 *   ToTensor + Normalize  regressor/human_shape/data/transforms/transforms.py:710-733  (clamp [0,1], (x - mean) / std)
 * The window corners are computed by the host exactly as transf_utils.py:41-56 does (float32 matrix inverse and
 * integer truncation; shapy_b200/preprocess.py mirrors it) and passed in the descriptor.
 *   images : device, all uint8 HxWx3 (RGB, row-major) images of the batch back to back
 *   descs  : device, one per output crop (several crops may name the same image)
 *   mean, stdv : host, 3 floats each
 *   out    : device (B, 3, size, size) fp32 */
typedef struct shapy_image_desc_t {
  long long offset;        /* byte offset of the image inside `images` */
  int height, width;       /* image extent */
  int ul_x, ul_y;          /* window upper-left corner (inclusive), may be negative */
  int br_x, br_y;          /* window bottom-right corner (exclusive), may exceed the image */
} shapy_image_desc_t;
int shapy_preprocess_forward(const unsigned char *images, const shapy_image_desc_t *descs, int batch, int size,
                             const float *mean, const float *stdv, float *out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * B2A attribute head (SURVEY.md 8f rank 2): betas -> attribute ratings with the male / female regressors.
 * Replaces regressor/human_shape/models/common/iterative_regressor.py:761-776 and
 * attributes/attributes/attributes_betas/polynomial.py:61-69,137-140 (degree-2 polynomial features + Linear).
 *   betas  : device (B, num_betas) fp32        gender : device (B) int32, 0 = male, 1 = female, other = row of zeros
 *   w_*    : device (num_outputs, num_betas + num_betas (num_betas + 1) / 2) fp32 row-major (Linear.weight)
 *   b_*    : device (num_outputs) fp32         out    : device (B, num_outputs) fp32 */
int shapy_b2a_forward(const float *betas, const int *gender, const float *w_male, const float *b_male,
                      const float *w_female, const float *b_female, int batch, int num_betas, int num_outputs, float *out,
                      void *stream);

/* A2B head (SURVEY.md 8f rank 2): attribute ratings (+ height / weight) -> betas, per gender.  Replaces
 * regressor/human_shape/models/common/iterative_regressor.py:837-850 around A2B.forward
 * (attributes/attributes/attributes_betas/a2b.py:278-279) for the `polynomial` (degree 2) and `linear` networks.
 *   feat_male / feat_female : device (B, num_features) fp32 -- the reference builds one feature vector per gender
 *                             (its default height / weight differ, iterative_regressor.py:793-836)
 *   gender : device (B) int32, 0 = male, 1 = female, other = row of zeros
 *   w_*    : device (num_betas, F) fp32 row-major, F = num_features (linear != 0) or num_features + num_features
 *            (num_features + 1) / 2 (degree-2 polynomial);  b_* : device (num_betas);  out : device (B, num_betas) */
int shapy_a2b_forward(const float *feat_male, const float *feat_female, const int *gender, const float *w_male,
                      const float *b_male, const float *w_female, const float *b_female, int batch, int num_features,
                      int num_betas, int linear, float *out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Evaluation metric (SURVEY.md 8f rank 3): translation-aligned point-to-point error through sparse point regressors
 * ("P2P-20k", also plain v2v with identity regressors).  Replaces regressor/human_shape/utils/metrics.py:368-456
 * (v2vhdError.__call__) and regressor/hbw_evaluation/evaluate_hbw.py:44-58,147-151.
 *   in_* / tg_* : device CSR (row_ptr int32 [P+1], col int32 [nnz], val fp32 [nnz]) of the P x V1 / P x V2 regressors
 *   input_vertices (B, V1, 3), target_vertices (B, V2, 3) : device fp32
 *   align : 1 = translate by mean(target points) - mean(input points) (metrics.py:431-439)
 *   error (B, P), mean_error (B) : device fp32      workspace : >= shapy_p2p_workspace_bytes(B, P) */
size_t shapy_p2p_workspace_bytes(int batch, int num_points);
int shapy_p2p_error(const int *in_row_ptr, const int *in_col, const float *in_val, const int *tg_row_ptr, const int *tg_col,
                    const float *tg_val, const float *input_vertices, const float *target_vertices, int batch, int num_points,
                    int num_input_vertices, int num_target_vertices, int align, float *error, float *mean_error, void *workspace,
                    size_t workspace_bytes, void *stream);

/* Vertex-to-vertex error between meshes of the SAME topology, translation aligned or not: PointError with
 * TranslationAlignment / NoAlignment, regressor/human_shape/utils/metrics.py:232-277, 335-366 (evaluation.py:192-224
 * `v2v_t` / `v2v`): est' = est + (mean(gt) - mean(est)); error[b][v] = |est'[b][v] - gt[b][v]|.
 * input / target: device (B, V, 3) fp32; error (B, V), mean_error (B); workspace >= shapy_p2p_workspace_bytes(B, V). */
int shapy_v2v_error(const float *input_vertices, const float *target_vertices, int batch, int num_verts, int align,
                    float *error, float *mean_error, void *workspace, size_t workspace_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SHAPY_B200_H_ */
