/*
 * p2m_b200.h — C ABI of libp2m_b200.so: the B200-native (sm_100a) MeshNet hot path of
 * hongsukchoi/Pose2Mesh_RELEASE.
 *
 * The reference has no FFI / operator registry: its boundary is the Python nn.Module contract
 *   models.meshnet.get_model(...) / Pose2Mesh.forward(x)              lib/models/meshnet.py:80-123
 *   models.backbones.cheby_graph_conv.graph_conv_cheby(x,cl,bn,L,..)  lib/models/backbones/cheby_graph_conv.py:5
 * (SURVEY.md §8b).  This header is the C boundary a binding (ctypes here, see INTEGRATION.md) sits
 * on: plain pointers and sizes, no torch types.  All `const float*` / `float*` data arguments are
 * DEVICE pointers owned by the caller unless a function name ends in `_host`.  Every function
 * returns 0 on success or a non-zero p2m_status; p2m_last_error() gives the message (thread-local).
 * Nothing here throws or aborts, and the library keeps no global mutable state (per-handle device
 * buffers and thread-local error / launch-count bookkeeping only), so one handle per device can be
 * driven from concurrent threads (nn.DataParallel, lib/core/base.py:108).  Entry points that touch
 * the device make the handle's device current for their own duration and restore the caller's.
 */
#ifndef P2M_B200_H_
#define P2M_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct p2m_model p2m_model_t;
typedef void* p2m_stream_t; /* cudaStream_t */

enum p2m_status {
  P2M_OK = 0,
  P2M_ERR_INVALID = 1,   /* bad argument / unsupported shape */
  P2M_ERR_CUDA = 2,      /* a CUDA runtime call or kernel launch failed */
  P2M_ERR_WORKSPACE = 3, /* workspace too small */
  P2M_ERR_NOGPU = 4      /* no usable sm_100 device */
};

enum p2m_precision {
  P2M_PREC_FP32_SIMT = 0, /* fp32 FFMA on CUDA cores (all shapes; the parity baseline)          */
  P2M_PREC_FP16X3_TC = 1  /* tcgen05 kind::f16, error-compensated 3-term fp16 split (~2^-21)    */
};

/* ---- the fixed mesh hierarchy + channel plan ---------------------------------------------------
 * Replaces what Pose2Mesh.__init__ derives from graph_L (meshnet.py:17-37,61-62): `n_levels`
 * Laplacians ordered fine -> coarse with the joint graph LAST and the second-coarsest mesh level
 * already removed (meshnet.py:35).  CSR arrays are HOST pointers (copied to the device here);
 * values are the float32 cast of the reference's float64 CSR (graph_utils.py:98-109).
 * `block_chans` is the concatenation of the per-block channel chains (meshnet.py:21-33), e.g. for
 * the SMPL plan {5,32,64,64, 64,128,256, ...}; `block_len[i]` is the length of chain i.           */
typedef struct {
  int32_t n_levels;
  const int32_t* level_size;        /* [n_levels] vertices per level                                  */
  const int32_t* const* rowptr;     /* [n_levels][V+1]                                                */
  const int32_t* const* colidx;     /* [n_levels][nnz]                                                */
  const float* const* values;       /* [n_levels][nnz]                                                */
  int32_t n_blocks;
  const int32_t* block_len;         /* [n_blocks]                                                     */
  const int32_t* block_chans;       /* [sum(block_len)]                                               */
  int32_t device;                   /* CUDA device ordinal                                            */
} p2m_model_desc_t;

/* Parameter / gradient tables: device pointers with the reference's state_dict layout
 * (SURVEY.md §8b): cl_w[i] is [Fout, 3*Fin] with column = fin*3 + k; bn_* entries are NULL for the
 * last conv (meshnet.py:52-53).  For gradients the same struct is used with d(.) pointers; bn_rm,
 * bn_rv, bn_nbt are ignored there.                                                                 */
typedef struct {
  float* fc_w;                 /* [V1*C1, J*C0]            */
  float* fc_b;                 /* [V1*C1]                  */
  float* const* cl_w;          /* [n_layers]               */
  float* const* cl_b;          /* [n_layers]               */
  float* const* bn_w;          /* [n_layers] gamma         */
  float* const* bn_b;          /* [n_layers] beta          */
  float* const* bn_rm;         /* [n_layers] running_mean  */
  float* const* bn_rv;         /* [n_layers] running_var   */
  int64_t* const* bn_nbt;      /* [n_layers] num_batches_tracked (may be NULL) */
} p2m_params_t;

int p2m_model_create(const p2m_model_desc_t* desc, p2m_model_t** out);
void p2m_model_destroy(p2m_model_t* m);
int p2m_model_num_layers(const p2m_model_t* m);
/* layer geometry: out[0]=level index, [1]=V, [2]=Fin, [3]=Fout, [4]=has_bn, [5]=relu */
int p2m_model_layer_info(const p2m_model_t* m, int layer, int32_t out[6]);
int p2m_model_set_precision(p2m_model_t* m, int precision);
/* Profiling: when enabled, the eval forward records a CUDA event pair (on the caller's stream) around
 * every conv layer; p2m_model_layer_times_ms returns the last forward's per-layer device times.      */
int p2m_model_set_profiling(p2m_model_t* m, int enable);
int p2m_model_layer_times_ms(p2m_model_t* m, float* out_ms, int n);
/* Every mbarrier wait of the tcgen05 kernels is time-bounded (2 s).  A kernel whose wait expired records the
 * wait's id in a per-handle status word the host can read without a copy; the NEXT entry point called on
 * the handle (and p2m_meshnet_forward_host itself, after its stream synchronisation) then fails with
 * P2M_ERR_CUDA and clears the word — results of a timed-out kernel are never returned silently.
 * p2m_debug_kernel_status device-synchronises and returns the word without clearing it (0 = clean).  */
int p2m_debug_kernel_status(p2m_model_t* m, int32_t* out);
/* Debug (libraries built with -DP2M_UMMA_TRACE only; P2M_ERR_INVALID otherwise): CTA 0 of this handle's
 * tcgen05 conv kernels logs (event << 48 | SM clock) into dev_buf [8][512] int64; NULL = off.        */
int p2m_debug_set_trace(p2m_model_t* m, void* dev_buf);
/* Debug / ablation: 1 (default) = T1 = L~x as a separate pass + conv with given T1; 0 = fully fused conv.   */
int p2m_debug_set_split_t1(p2m_model_t* m, int enable);
/* Debug / ablation: 1 (default) = in eval mode the 128->64 conv's epilogue produces the 64->3 head's projections
 * itself (the 64-wide activation is never written); 0 = the two layers run separately.                         */
int p2m_debug_set_fuse_head(p2m_model_t* m, int enable);
/* Padding-vertex elision: the isolated padding vertices of each level (the fake nodes of the reference's binary-tree
 * reorder, lib/coarsening.py:214-258) go through a plain GEMM with the combined weights W0 + c W1 + (2c^2-1) W2, the
 * connected rows through the conv on index-list tiles.  Same results up to fp32 association.  1 (default) = on levels
 * where at least 40 % of the rows are isolated, 2 = wherever the tile families exist, 0 = off.                       */
int p2m_debug_set_elide_padding(p2m_model_t* m, int enable);
/* Eval mode, on the elided levels: both children of a fake vertex are fake and carry identical values, so only one
 * representative per class of identical isolated rows is computed and the output rows of the others are filled from
 * it at the end; p2m_meshnet_forward_vertices (which returns connected rows only) computes no isolated row at all.
 * 1 (default) = on, 0 = every isolated row is computed.  Training always computes every row (BatchNorm statistics). */
int p2m_debug_set_dedup_padding(p2m_model_t* m, int enable);
/* Backward, tensor-core layers: 1 (default) = the weight gradient is formed from the Chebyshev basis of the GRADIENT
 * (sum_rows dz (x) T_k(x) = sum_rows T_k(dz) (x) x, L~ symmetric), re-using the L~dz the backward-data pass computes;
 * 0 = from the basis of the layer input, rebuilt on chip with its 2-hop halo.  Same result up to fp32 association. */
int p2m_debug_set_dw_swap(p2m_model_t* m, int enable);

/* Bytes of device workspace p2m_meshnet_forward needs for batch B.  In training mode the workspace
 * also carries what p2m_meshnet_backward reads, so it must stay alive and untouched in between.   */
size_t p2m_meshnet_workspace_bytes(const p2m_model_t* m, int batch, int training);
size_t p2m_meshnet_backward_scratch_bytes(const p2m_model_t* m, int batch);

/* Pose2Mesh.forward (meshnet.py:80-117): x [B, J, Cin] -> y [B, V0, Cout].
 * training=0: BatchNorm uses running stats (folded into the conv epilogue).
 * training=1: batch statistics, running stats updated (momentum 0.1, eps 1e-5), activations kept. */
int p2m_meshnet_forward(p2m_model_t* m, const p2m_params_t* params, const float* x, float* y, int batch,
                        int training, void* workspace, size_t workspace_bytes, p2m_stream_t stream);

/* Fused output gather (SURVEY.md §8a row a9): the callers' `pred[:, perm_reverse[:n_real], :]`
 * (lib/core/base.py:130,201; demo/run.py:170) folded into the head layer's store.  `vertex_of_slot` (HOST,
 * int32[n_slots]) is perm_reverse[:n_real]; p2m_meshnet_forward_vertices then writes y_vertices [B, n_slots, Cout]
 * (eval mode) instead of the padded [B, V0, Cout].                                                    */
int p2m_model_set_output_gather(p2m_model_t* m, const int32_t* vertex_of_slot, int n_slots);
int p2m_meshnet_forward_vertices(p2m_model_t* m, const p2m_params_t* params, const float* x, float* y_vertices,
                                 int batch, void* workspace, size_t workspace_bytes, p2m_stream_t stream);

/* Backward of the training forward above.  dy [B,V0,Cout]; dx [B,J,Cin] (may be NULL).  Gradients
 * are WRITTEN (not accumulated) into `grads`.                                                     */
int p2m_meshnet_backward(p2m_model_t* m, const p2m_params_t* params, const p2m_params_t* grads, const float* x,
                         const float* dy, float* dx, int batch, void* workspace, size_t workspace_bytes,
                         void* scratch, size_t scratch_bytes, p2m_stream_t stream);

/* End-to-end inference with HOST buffers (pageable or pinned): H2D of x, forward (eval), D2H of y,
 * stream-synchronised on return.  `workspace` must additionally hold x and y
 * (p2m_meshnet_workspace_bytes(...) + p2m_meshnet_host_io_bytes(...)).                             */
size_t p2m_meshnet_host_io_bytes(const p2m_model_t* m, int batch);
int p2m_meshnet_forward_host(p2m_model_t* m, const p2m_params_t* params, const float* x_host, float* y_host,
                             int batch, void* workspace, size_t workspace_bytes, p2m_stream_t stream);
/* Same with the fused output gather (p2m_model_set_output_gather): y_vertices_host is [B, n_slots, Cout], i.e. what
 * the reference's callers keep of a mesh (lib/core/base.py:130,201; demo/run.py:170) — 6890 of the 12288 rows.   */
int p2m_meshnet_forward_vertices_host(p2m_model_t* m, const p2m_params_t* params, const float* x_host,
                                      float* y_vertices_host, int batch, void* workspace, size_t workspace_bytes,
                                      p2m_stream_t stream);

/* ---- single Chebyshev graph convolution ----------------------------------------------------------
 * graph_conv_cheby (cheby_graph_conv.py:5-42) on hierarchy level `level`:
 *   y = act( bn( [T0|T1|T2] W^T + b ) ),  T0=x, T1=L~x, T2=2L~T1-x,   x [B,V,Fin] -> y [B,V,Fout]
 * bn_mode 0: none; 1: eval affine from running stats; 2: batch statistics (running stats updated,
 *            save_mean/save_invstd [Fout] written if non-NULL).                                    */
typedef struct {
  int32_t level, batch, fin, fout;
  const float* x;
  const float* weight;      /* [Fout, 3*Fin], column = fin*3 + k */
  const float* bias;        /* [Fout]                            */
  int32_t bn_mode;
  const float* bn_weight;
  const float* bn_bias;
  float* bn_running_mean;
  float* bn_running_var;
  int64_t* bn_num_batches_tracked;
  float* save_mean;
  float* save_invstd;
  int32_t relu;
  float* y;
} p2m_conv_fwd_args_t;

size_t p2m_cheb_conv_workspace_bytes(const p2m_model_t* m, int level, int batch, int fin, int fout);
int p2m_cheb_conv_fwd(p2m_model_t* m, const p2m_conv_fwd_args_t* a, void* workspace, size_t workspace_bytes,
                      p2m_stream_t stream);

/* Backward of the linear part  z = [T0|T1|T2] W^T + b  (BatchNorm / ReLU backward are the caller's):
 * dz [B,V,Fout] -> dx [B,V,Fin] (may be NULL), dweight [Fout,3Fin], dbias [Fout].                  */
typedef struct {
  int32_t level, batch, fin, fout;
  const float* x;
  const float* weight;
  const float* dz;
  float* dx;
  float* dweight;
  float* dbias;
} p2m_conv_bwd_args_t;
int p2m_cheb_conv_bwd(p2m_model_t* m, const p2m_conv_bwd_args_t* a, void* workspace, size_t workspace_bytes,
                      p2m_stream_t stream);

/* ---- the step in front of MeshNet (SURVEY.md §8 row f1) --------------------------------------------
 * FlatPose2Mesh.forward (lib/models/pose2mesh_net.py:16-22) in eval mode: PoseNet, the 2-D -> 3-D pose lifter
 * (lib/models/posenet.py:41-87: Linear(2J,H), `num_stage` residual stages of BN-ReLU-Linear(H,H)-BN-ReLU-Linear(H,H),
 * Linear(H,3J); running-stat BatchNorm, dropout off), and pose_combine = cat(pose2d, pose3d / 1000) [B, J, 5],
 * MeshNet's input.  All pointers are device pointers with the reference's state_dict shapes.               */
typedef struct {
  const float* w1_w; const float* w1_b;                                     /* [H, H], [H]   */
  const float* w2_w; const float* w2_b;
  const float* bn1_w; const float* bn1_b; const float* bn1_rm; const float* bn1_rv;   /* [H] each */
  const float* bn2_w; const float* bn2_b; const float* bn2_rm; const float* bn2_rv;
} p2m_posenet_stage_t;
typedef struct {
  int32_t num_joint, hidden, num_stage;
  const float* w1_w; const float* w1_b;        /* [H, 2J], [H]  */
  const float* w2_w; const float* w2_b;        /* [3J, H], [3J] */
  const p2m_posenet_stage_t* stages;           /* [num_stage] (host array of device pointers) */
} p2m_posenet_params_t;
size_t p2m_posenet_workspace_bytes(int batch, int hidden);
/* pose2d [B, 2J] -> pose3d [B, 3J]; pose_combine (optional) [B, J, 5].  Enqueued on `stream` of the current device. */
int p2m_posenet_forward(const p2m_posenet_params_t* params, const float* pose2d, float* pose3d, float* pose_combine,
                        int batch, void* workspace, size_t workspace_bytes, p2m_stream_t stream);

/* ---- the steps either side of the model in the reference's callers (SURVEY.md §8 row f2) ----------
 * Joint regression (lib/core/base.py:131,204; demo/run.py:171): joints [B, n_joint, C] = joint_regressor
 * [n_joint, n_vertex] @ vertices [B, n_vertex, C] (C <= 4), on the gathered vertices of
 * p2m_meshnet_forward_vertices.                                                                        */
int p2m_regress_joints(const float* joint_regressor, const float* vertices, float* joints, int batch, int n_joint,
                       int n_vertex, int chans, p2m_stream_t stream);
/* The demo's input normalisation (demo/run.py:150-158): joints_px [B, J, 2] in image pixels -> pose2d [B, J, 2],
 * zero mean / unit std per pose and coordinate in the aspect-preserving box of the (input_h, input_w) network input
 * (cfg.MODEL.input_shape = (384, 288)).  truncate_like_int_input = 1 reproduces the reference on INTEGER joint
 * arrays (demo/h36m_joint_input.npy is int64: the transformed coordinates are truncated when written back). */
int p2m_normalize_pose2d(const float* joints_px, float* pose2d, int batch, int n_joint, int input_h, int input_w,
                         int truncate_like_int_input, p2m_stream_t stream);

/* ---- the demo's camera fit (SURVEY.md §8 row f5; demo/run.py:149-189, lib/models/project_net.py) --------------
 * The projection target: joints_px [B, J, 2] (J <= 32) -> out_px [B, J, 2], the joints in pixels of a res_w x res_h
 * patch cut around the box process_bbox(get_bbox(joints), aspect_ratio, scale) (the demo: 500 x 500, 1.0, 1.25), and
 * out_bbox [B, 4] = that box [x, y, w, h] (the demo's bbox1).  truncate_like_int_input as in p2m_normalize_pose2d.   */
int p2m_crop_pose2d(const float* joints_px, float* out_px, float* out_bbox, int batch, int n_joint, int res_w, int res_h,
                    float aspect_ratio, float scale, int truncate_like_int_input, p2m_stream_t stream);
/* The weak-perspective camera out = (p[:, :2] + c[1:]) * c[0] * crop_size / 2 + crop_size / 2 fitted per person to
 * target_px [B, J, 2] by `iters` steps of mean L1 loss + Adam (torch.optim.Adam defaults; lr 0.1, 0.05 from step 502,
 * 0.001 from step 1002), starting from cam_init [B, 3].  joints3d [B, J, joint_stride] (x, y first; joint_stride >= 2),
 * J <= 32.  Writes cam_out [B, 3] and loss_out [B], the L1 loss of the final camera.  One warp per person.          */
int p2m_fit_camera(const float* joints3d, const float* target_px, const float* cam_init, float* cam_out, float* loss_out,
                   int batch, int n_joint, int joint_stride, double crop_size, int iters, p2m_stream_t stream);

/* ---- the mesh losses (SURVEY.md §8 row f3; lib/core/loss.py:10-23,62-114) ---------------------------
 * One pass over (mesh, face): sums[0] = sum of the NormalVectorLoss terms, sums[1] = sum of the EdgeLengthLoss terms
 * over (B, 3 n_face) (fp64, device; the losses are sums / (3 B n_face)).  If grad_out [B, n_vertex, 3] is given it
 * receives  grad_scale[0] * d sums[0] / d coord_out + grad_scale[1] * d sums[1] / d coord_out  (grad_scale: device
 * float[2], i.e. upstream gradient / (3 B n_face)).  faces: device int32 [n_face, 3].                    */
int p2m_mesh_losses(const float* coord_out, const float* coord_gt, const int32_t* faces, int batch, int n_vertex,
                    int n_face, const float* grad_scale, double* sums, float* grad_out, p2m_stream_t stream);
/* CoordLoss: *sum = sum |pred * valid - target * valid| over n elements (valid may be NULL = ones, else same shape);
 * grad_out (optional, n floats) = grad_scale[0] * sign(.) * valid.                                        */
int p2m_coord_loss(const float* pred, const float* target, const float* valid, int64_t n, const float* grad_scale,
                   double* sum, float* grad_out, p2m_stream_t stream);

/* ---- host-side graph baking helper (CPU; no device work) -------------------------------------------
 * One level of the reference's greedy heavy-edge matching (lib/coarsening.py:153-211, HEM_one_level),
 * entries sorted by (row, col); returns the number of clusters (or -1).  Driven by
 * pose2mesh_release_b200/graph.py, which replaces build_coarse_graphs (lib/graph_utils.py:75-95).   */
int32_t p2m_graph_match_level(int64_t nnz, const int32_t* rows, const int32_t* cols, const double* vals,
                              const int64_t* visit_order, const double* weights, int32_t* cluster_out);

/* ---- misc ----------------------------------------------------------------------------------------*/
const char* p2m_last_error(void);
const char* p2m_version(void);
/* Number of kernels this library launched on behalf of the calling thread since the last reset.    */
int64_t p2m_launch_count(void);
void p2m_launch_count_reset(void);

#ifdef __cplusplus
}
#endif
#endif /* P2M_B200_H_ */
