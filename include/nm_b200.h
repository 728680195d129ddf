/* nm_b200 — C ABI of the B200-native Neural Marionette keypoint-detection hot path.
 *
 * The reference (jinseokbae/neural_marionette) is pure Python over torch.nn: it has no FFI / plugin
 * interface.  The drop-in boundary is therefore its Python class surface (SURVEY.md §8b); this header is the
 * thin C ABI those classes call.  Each entry point names the reference code it replaces (file:line under the
 * reference tree).  Conventions:
 *   - every pointer is a DEVICE pointer unless the name says `host`; no allocation inside the library;
 *     scratch memory is caller-provided (`*_workspace_bytes` gives the size);
 *   - `stream` is a cudaStream_t passed as void*; the call only enqueues work on it (re-entrant per stream);
 *   - return value 0 = ok, non-zero = error, message via nm_last_error() (thread-local);
 *   - activations between kernels are fp16 channels-last (n, D, H, W, C) ("act" below); tensors that cross
 *     the Python API (occupancy grids, heat-maps, keypoints, gaussians, reconstructions) are fp32 in the
 *     reference's NCDHW layout.
 */
#ifndef NM_B200_H
#define NM_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

const char* nm_last_error(void);
int nm_version(void);
/* sm_100a check: returns 0 when the current device can run the kernels */
int nm_device_supported(void);

/* ---- voxelization ------------------------------------------------------------------------------------
 * utils/dataset_utils.py:21-31 `voxelize(pos_coords, output_shape, is_binarized=True)`.
 * points: (n_frames, n_points, 3) float64 (points_are_f64=1, what episodic_normalization returns) or float32.
 * grid_out: (n_frames, G, G, G) fp32, fully overwritten (0/1).  err_flag (optional int) is OR-ed with 1 when a
 * point falls outside [-1, 1) (numpy would wrap / raise there). */
int nm_voxelize(const void* points, int points_are_f64, int n_frames, int n_points, int grid_size,
                float* grid_out, int* err_flag, void* stream);
/* utils/dataset_utils.py:9-19 + :21-31 fused: raw fp32 clips (n_clips, T, n_points, 3) -> clip-global bbox
 * normalisation (fp32 op order of the reference, float64 translation) -> occupancy (n_clips*T, G, G, G).
 * bounds_out (optional): (n_clips, 6) fp32 = bmin xyz, bmax xyz. */
size_t nm_normalize_voxelize_workspace_bytes(int n_clips);
int nm_normalize_voxelize(const float* raw_points, int n_clips, int T, int n_points, int grid_size, float scale,
                          double x_trans, double z_trans, float* grid_out, float* bounds_out, void* workspace,
                          int* err_flag, void* stream);

/* ---- convolutions ------------------------------------------------------------------------------------
 * nn.Conv3d weight (Cout, Cin, k, k, k) fp32 -> tensor-core operand layout [k^3][Cout][Cin] fp16. */
int nm_pack_conv_weights(const float* weight, void* packed, int Cout, int Cin, int k, void* stream);
/* modules/vox_modules.py:12,26,30,39,53; model/kypt_detector.py:429,435,444,450 — nn.Conv3d with
 * (k in {1,3}, stride 1, pad (k-1)/2) or (k 2, stride 2).  tcgen05 implicit GEMM; x, out: act. */
int nm_conv3d_tc(const void* x, const void* packed_w, const float* bias, void* out, int n, int D, int H, int W,
                 int Cin, int Cout, int k, int stride, float* stats_partial, void* stream);
/* GroupNorm statistics fused into the conv epilogue: when nm_conv3d_stats_chunks(...) > 0 the conv can write
 * per-sample partial (sum, sum of squares) of its fp32 output to stats_partial [n][chunks][Cout][2]; feed them
 * to nm_groupnorm_finalize instead of re-reading the tensor with nm_groupnorm_scale_shift. */
int nm_conv3d_stats_chunks(int n, int D, int H, int W, int Cin, int Cout, int k, int stride);
/* Same conv with the producing layer's GroupNorm (+LeakyReLU) fused into the operand path: the input is the RAW
 * output of the previous conv and x <- act(x * in_scale[n][c] + in_shift[n][c]) is applied to each halo slice in
 * shared memory before the MMAs read it (zero padding preserved), so the activated tensor is never written to HBM
 * (replaces the nn.GroupNorm + nn.LeakyReLU between two convs, modules/vox_modules.py:26-32,
 * model/kypt_detector.py:429-453).  Only where nm_conv3d_can_fuse_input(...) == 1. */
int nm_conv3d_can_fuse_input(int n, int D, int H, int W, int Cin, int Cout, int k, int stride);
int nm_conv3d_tc_fused(const void* x, const void* packed_w, const float* bias, void* out, int n, int D, int H, int W,
                       int Cin, int Cout, int k, int stride, const float* in_scale, const float* in_shift, int in_act,
                       float* stats_partial, void* stream);
/* same contract on CUDA cores from the raw fp32 weight; on-device cross-check of nm_conv3d_tc */
int nm_conv3d_direct(const void* x, const float* weight, const float* bias, void* out, int n, int D, int H, int W,
                     int Cin, int Cout, int k, int stride, int pad, void* stream);
/* modules/vox_modules.py:68 nn.ConvTranspose3d(k 2, stride 2); weight: the (Cin, Cout, 2, 2, 2) fp32 parameter
 * permuted to tap-major (8, Cin, Cout) */
int nm_conv_transpose3d_k2s2(const void* x, const float* weight, const float* bias, void* out, int n, int D, int H,
                             int W, int Cin, int Cout, void* stream);
/* k3 conv whose input is the 2x trilinear up-sampling (align_corners = False) of x_lo (n, D/2, H/2, W/2, Cin): the
 * up-sampled tensor is never written - the halo slices of the tcgen05 kernel are interpolated in shared memory from
 * low-resolution planes (reference: nn.Upsample(scale_factor=2, mode='trilinear') + nn.Conv3d(k3) in
 * build_voxel_decoder, model/kypt_detector.py:385-396).  (D, H, W) is the OUTPUT extent.  Optional fused input
 * transform act(x_lo*in_scale+in_shift) and fused GroupNorm statistics as for nm_conv3d_tc_fused (chunks from
 * nm_conv3d_stats_chunks(n, D, H, W, Cin, Cout, 3, 1)).  packed_w from nm_pack_conv_weights. */
int nm_conv3d_up2x_supported(int n, int D, int H, int W, int Cin, int Cout);
int nm_conv3d_tc_up2x(const void* x_lo, const void* packed_w, const float* bias, void* out, int n, int D, int H, int W,
                      int Cin, int Cout, const float* in_scale, const float* in_shift, int in_act,
                      float* stats_partial, void* stream);

/* Pointwise-shaped convolutions with Cin in {32, 64} on mma.sync, organised around the memory pipe: Conv3d(k2, s2) of
 * Pool3DBlock (modules/vox_modules.py:49-61) and the 1x1 skip convolution of Res3DBlock (modules/vox_modules.py:35-38);
 * shapes: nm_conv3d_pw_supported.  Optional fused input transform
 *     input = act(x*in_scale + in_shift) [+ x2*in_scale2 + in_shift2]
 * (scales/shifts (n, Cin) fp32: a producer's GroupNorm folded to scale/shift; in_act != 0: LeakyReLU 0.01 on the first
 * term; x2: a second tensor of x's shape - the other branch of a Res3DBlock, modules/vox_modules.py:40-47 - added as
 * is when in_scale2 is null) and fused GroupNorm statistics of the output: stats_partial [n][chunks][Cout][2] for
 * nm_groupnorm_finalize, chunks = nm_conv3d_pw_stats_chunks(...).
 * packed_w comes from nm_pack_conv_pw_weights (weight: the nn.Conv3d (Cout, Cin, k, k, k) fp32 tensor). */
int nm_conv3d_pw_supported(int n, int D, int H, int W, int Cin, int Cout, int k, int stride);
int nm_conv3d_pw_dual_supported(int n, int D, int H, int W, int Cin, int Cout, int k, int stride);  /* x2 allowed */
int nm_conv3d_pw_stats_chunks(int n, int D, int H, int W, int Cin, int Cout, int k, int stride);
size_t nm_conv3d_pw_packed_bytes(int Cin, int Cout, int k);
int nm_pack_conv_pw_weights(const float* weight, int Cin, int Cout, int k, void* packed, void* stream);
int nm_conv3d_pw(const void* x, const void* packed_w, const float* bias, void* out, int n, int D, int H, int W, int Cin,
                 int Cout, int k, int stride, const float* in_scale, const float* in_shift, int in_act, const void* x2,
                 const float* in_scale2, const float* in_shift2, float* stats_partial, void* stream);

/* ConvTranspose3d(k2, s2) with Cin = 32 on mma.sync (Upsample3DBlock, modules/vox_modules.py:63-75); weight is the
 * nn.ConvTranspose3d (Cin, Cout, 2, 2, 2) fp32 tensor; x (n, D, H, W, Cin) -> out (n, 2D, 2H, 2W, Cout); optional
 * GroupNorm statistics of the output as in nm_conv3d_pw. */
int nm_conv_transpose3d_pw_supported(int n, int D, int H, int W, int Cin, int Cout);
int nm_conv_transpose3d_pw_stats_chunks(int n, int D, int H, int W, int Cin, int Cout);
size_t nm_conv_transpose3d_pw_packed_bytes(int Cin, int Cout);
int nm_pack_conv_transpose3d_pw_weights(const float* weight, int Cin, int Cout, void* packed, void* stream);
int nm_conv_transpose3d_pw(const void* x, const void* packed_w, const float* bias, void* out, int n, int D, int H, int W,
                           int Cin, int Cout, float* stats_partial, void* stream);

/* First layer: add_coord_channels (utils/kypt_detector_utils.py:4-26) + Conv3d(1+3, Cout, k5, pad 2)
 * (model/kypt_detector.py:266).  occ: (n, G, G, G) fp32; weight (Cout, 4, 5, 5, 5) fp32; out: act (n,G,G,G,Cout).
 * `tables` is built once per weight set by nm_first_conv_prepare. linspace: torch.linspace(-1,1,G) fp32. */
size_t nm_first_conv_tables_bytes(int Cout);
int nm_first_conv_prepare(const float* weight, int Cout, void* tables, void* stream);
int nm_first_conv_stats_chunks(int G);
/* stats_partial: null, or [n][nm_first_conv_stats_chunks(G)][Cout][2] per-channel (sum, sum of squares) partials of
 * the output for nm_groupnorm_finalize (the GroupNorm that follows, modules/vox_modules.py:14). */
int nm_first_conv_k5(const float* occ, const void* tables, const float* bias, const float* linspace, int n, int G,
                     int Cout, void* out, float* stats_partial, void* stream);

/* ---- GroupNorm / pointwise ---------------------------------------------------------------------------
 * nn.GroupNorm(C//16, C) statistics (modules/vox_modules.py:14,...) folded to per-(sample, channel)
 * scale/shift: y = x*scale + shift.  x: act (n, S, C). */
size_t nm_gn_workspace_bytes(int n, int S, int C);
/* mean_rstd (optional, (n, groups, 2)) and xsum (optional, (n, C) per-channel sums): the statistics the training path
 * keeps for nm_groupnorm_backward. */
int nm_groupnorm_scale_shift(const void* x, int n, int S, int C, int groups, const float* gamma, const float* beta,
                             float eps, float* scale, float* shift, void* workspace, float* mean_rstd, float* xsum,
                             void* stream);
int nm_groupnorm_finalize(const float* partial, int n, int S, int C, int groups, int chunks, const float* gamma,
                          const float* beta, float eps, float* scale, float* shift, float* mean_rstd, float* xsum,
                          void* stream);
/* out = act1(x1*a1+b1) + (x2*a2+b2 | x2 | nothing); act1: 0 none, 1 LeakyReLU(0.01).
 * Basic/Pool/Upsample blocks, Res3DBlock sums (vox_modules.py:44-47), HG skip adds (:111-118). */
int nm_affine_act(const void* x1, const float* a1, const float* b1, int act1, const void* x2, const float* a2,
                  const float* b2, void* out, int n, int S, int C, void* stream);
/* nn.Upsample(scale 2, trilinear, align_corners=False) (kypt_detector.py:427,441) of act1(x*a+b) (a,b optional) */
int nm_upsample2x(const void* x, const float* a, const float* b, int act, void* out, int n, int D, int H, int W, int C,
                  void* stream);
int nm_ndhwc_to_ncdhw_f32(const void* x, float* out, int n, int S, int C, long long in_sample_stride, void* stream);
int nm_ncdhw_f32_to_ndhwc(const float* x, void* out, int n, int S, int C, void* stream);
/* seq.mean(dim=1) (kypt_detector.py:312): (n_clips, T, S) fp32 -> (n_clips, S) */
int nm_mean_over_frames(const float* seq, float* out, int n_clips, int T, long long S, void* stream);
/* decoder tail: GN-apply + LeakyReLU + Conv3d(32,1,k1) + sigmoid(sharp*(tanh(x)+first_frame-trans))
 * (kypt_detector.py:453-457,:410) and, when `target` is given, the per-frame mean BCE (:91-92).
 * bias_dev (optional, here and in the two backward entry points): device pointer to the 1x1 conv's bias - overrides
 * `bias`, so that a training loop never reads the updated parameter back to the host. */
size_t nm_final_recon_workspace_bytes(int n);
int nm_final_recon(const void* x, const float* a, const float* b, const float* w, float bias, const float* bias_dev,
                   const float* first_frame,
                   int frames_per_clip, float sharpness, float translation, float* recon, const float* target,
                   float* bce_mean, void* workspace, int n, int S, int C, void* stream);
/* get_volume_fitting_loss('chamfer') (utils/kypt_detector_utils.py:141-157): per-frame value, (n) fp32 */
size_t nm_chamfer_workspace_bytes(int n);
int nm_chamfer_vol_fit(const float* seq, const float* keypoints, const float* linspace, int n, int K, int G,
                       float* out, void* workspace, void* stream);

/* ---- heat-map heads / soft-argmax / Gaussian render --------------------------------------------------
 * mode 0: heat = LeakyReLU(conv1x1(feature))                        (kypt_detector.py:315: ST head)
 * mode 1: heat = Softplus(pw0*LeakyReLU(conv1x1(feature)) + pw1*prev[clip] + pb)   (:336-343)
 *         keypoints = extract_keypoints_from_heatmap(heat)           (utils/kypt_detector_utils.py:28-55)
 *         gaussians = extract_gaussian_map_from_keypoints(...)       (:57-90), optional
 * feature: act (n, g^3, C); w1 (K, C); prev (n/frames_per_clip, K, g^3); heat/gaussians (n, K, g^3); keypoints (n,K,4).
 * heat_mean (optional, (n,K)): per-keypoint heat-map mean = input of get_keypoint_sparsity_loss (:92-103).
 * gauss_width = 2*(sigma/g)^2 computed by the caller in double.
 * prop_dev (optional, also in nm_heatmap_head_backward): device pointer to (pw0, pw1, pb) - overrides the by-value copies.
 * K <= 64 here, in nm_gaussian_render / nm_decoder_adjust and in their backward entry points (K <= 24 runs the tuned
 * kernels). */
int nm_heatmap_head(const void* feature, const float* w1, const float* b1, int n, int g, int C, int K, int mode,
                    const float* prev, int frames_per_clip, float pw0, float pw1, float pb, const float* prop_dev,
                    const float* linspace, float gauss_width, float* heat, float* keypoints, float* gaussians, float* heat_mean,
                    void* stream);
int nm_gaussian_render(const float* keypoints, int n, int K, int g, const float* linspace, float gauss_width,
                       float* gaussians, void* stream);
/* adjust_combined_representation (kypt_detector.py:381,404-408): 1x1 conv over cat[gauss_t, first_feature,
 * gauss_0, coords] + LeakyReLU, with the clip-constant part hoisted.  first_feature: act (n_clips, g^3, 128);
 * keypoints (n, K, 4) or gaussians (n, K, g^3) with n = n_clips*frames_per_clip; base_ws:
 * nm_decoder_adjust_workspace_bytes(n_clips, g) bytes (the per-clip fp32 base + packed weight fragments);
 * out: act (n, g^3, 128). */
size_t nm_decoder_adjust_workspace_bytes(int n_clips, int g);
int nm_decoder_adjust(const void* first_feature, const float* keypoints, const float* gaussians, const float* weight,
                      const float* bias, int n_clips, int frames_per_clip, int g, int K, const float* linspace,
                      float gauss_width, float* base_ws, void* out, void* stream);

/* ---- HSVRNN latent dynamics --------------------------------------------------------------------------
 * Weights are passed TRANSPOSED ([in][out], fp32) so that output columns are contiguous. */
typedef struct nm_hsvrnn_weights {
  const float *post0_wt, *post0_b, *post2_wt, *post2_b;       /* extract_post_dist  (hsvrnn_bvh.py:29-34) */
  const float *prior0_wt, *prior0_b, *prior2_wt, *prior2_b;   /* extract_prior_dist (:35-40) */
  const float *root0_wt, *root0_b, *root2_wt, *root2_b;       /* root_intensity_decoder (:41-47) */
  const float *joint0_wt, *joint0_b, *joint2_wt, *joint2_b;   /* joint_matrix_decoder (:49-54) */
  const float *gru_ih_wt, *gru_hh_wt, *gru_ih_b, *gru_hh_b;   /* kypt_rnn_cell (:57-58), gate order r,z,n */
} nm_hsvrnn_weights;
/* One time step (hsvrnn_bvh.py:89-135 posterior / :208-225 prior).  `w` is a HOST pointer to the struct.
 * h_in/h_out (B,512); kp (B,4K) detected keypoints (posterior); eps (S,B,128) standard-normal draws;
 * offset (B,K,3); order/parents (K) int32 = priority.indices / parents; kp_out (B,4K) decoded keypoints fed to
 * the GRU; optional outputs: z_out (B,128), R_out (B,K,9), post_out / prior_out (B,256) = mean | std.
 * 0 < K <= 64 here and in every nm_hsvrnn_* entry point (K <= 24 runs the tuned kernels); S <= 16. */
int nm_hsvrnn_step(const nm_hsvrnn_weights* w, const float* h_in, const float* kp, const float* eps, const float* offset,
                   const int* order, const int* parents, int B, int K, int S, int posterior, float* h_out,
                   float* kp_out, float* z_out, float* R_out, float* post_out, float* prior_out, void* stream);
/* nm_hsvrnn_step that also records, in pick_out (B) int32 (nullable), which of the S samples each element fed to the GRU.
 * The arithmetic is that of nm_hsvrnn_step. */
int nm_hsvrnn_step_record(const nm_hsvrnn_weights* w, const float* h_in, const float* kp, const float* eps,
                          const float* offset, const int* order, const int* parents, int B, int K, int S, int posterior,
                          float* h_out, float* kp_out, float* z_out, float* R_out, float* post_out, float* prior_out,
                          int* pick_out, void* stream);
/* ---- stage-2 training: backward of HSVRNNBVH.encode (hsvrnn_bvh.py:67-156), one call per step from t = T-1 down to 0.
 * wt: the weights as for nm_hsvrnn_step ([in][out]); w: the same struct pointing at the fp32 parameters in their own
 * [out][in] layout (nn.Linear.weight, GRUCell.weight_ih / weight_hh).  Saved from the forward of step t: h (B,512) = h_t,
 * kp (B,4K), eps (S,B,128), pick (B) from nm_hsvrnn_step_record, f (B,4K) / z (B,128) / R (B,K,9) the step's kp_out /
 * z_out / R_out, offset (B,K,3).  Incoming gradients: dh_next (B,512) of h_{t+1}, already including the external gradient
 * of h_{t+1}; nullable: dh_ext (B,512) the external gradient of h_t, df (B,4K), dR (B,K,9), dz (B,128), dpost / dprior
 * (B,256) of (mean | std).  Outputs: dh_out (B,512) the full gradient of h_t; doffset (B,K,3) is ACCUMULATED into; rows
 * (B x nm_hsvrnn_backward_workspace_bytes(1, 1) bytes) is this step's slice of the workspace, read later by
 * nm_hsvrnn_weight_grads.  No gradient flows to kp. */
size_t nm_hsvrnn_backward_workspace_bytes(int B, int T);
int nm_hsvrnn_step_backward(const nm_hsvrnn_weights* wt, const nm_hsvrnn_weights* w, const float* h, const float* kp,
                            const float* eps, const int* pick, const float* f, const float* z, const float* R,
                            const float* offset, const int* order, const int* parents, int B, int K, int S,
                            const float* dh_next, const float* dh_ext, const float* df, const float* dR, const float* dz,
                            const float* dpost, const float* dprior, float* dh_out, float* doffset, float* rows,
                            void* stream);
/* Gradients of the parameters in their own layouts ([out][in] weights), fully overwritten. */
typedef struct nm_hsvrnn_grads {
  float *post0_w, *post0_b, *post2_w, *post2_b, *prior0_w, *prior0_b, *prior2_w, *prior2_b;
  float *root0_w, *root0_b, *root2_w, *root2_b, *joint0_w, *joint0_b, *joint2_w, *joint2_b;
  float *gru_ih_w, *gru_hh_w, *gru_ih_b, *gru_hh_b;
  float* init_state;     /* (512): sum over b of dh_0 */
  float* offset_param;   /* (K,3) or null (offset_param frozen) */
} nm_hsvrnn_grads;
/* After the reverse loop: one launch computes every weight / bias gradient over the T*B rows (r = t*B + b) of `rows`
 * (the whole workspace) in a fixed order - no atomics, bit-reproducible - plus the init-state gradient from dh0 (B,512)
 * and, when g->offset_param is set, the offset_param gradient from offset / doffset (B,K,3) and offset_param (K,3).
 * h (T+1,B,512) or at least its first T*B rows, kp / f (T,B,4K), z (T,B,128): the forward's per-step tensors. */
int nm_hsvrnn_weight_grads(const float* rows, const float* h, const float* kp, const float* f, const float* z,
                           const float* dh0, const float* offset, const float* doffset, const float* offset_param, int B,
                           int T, int K, const nm_hsvrnn_grads* g, void* stream);
/* extract_kypt_from_latent_and_state (hsvrnn_bvh.py:255-286): dec_in (B, 640) -> flat (B, 4K), R (B, K, 9) */
int nm_hsvrnn_decode_pose(const nm_hsvrnn_weights* w, const float* dec_in, const float* offset, const int* order,
                          const int* parents, int B, int K, float* flat_out, float* R_out, void* stream);
/* get_offset (hsvrnn_bvh.py:236-253): keypoints (B,T,K,4) -> (B,K,3) */
int nm_hsvrnn_bone_offsets(const float* keypoints, const int* parents, const float* offset_param, int B, int T, int K,
                           float* out, void* stream);

/* ---- consumers of the path's outputs (SURVEY.md §8f#4) -----------------------------------------------
 * utils/eval_utils.py:29-56 `voxel_chamfer_distance`: per-frame symmetric chamfer distance between the occupied
 * voxels of gt (n, G, G, G; non-zero = occupied) and of recon (>= 0.5 = occupied; binarised IN PLACE when
 * binarize_recon != 0, as :37-38 do), coordinates idx / ((G-1)/2) - 1.  out (n) fp32; a frame whose gt or recon
 * is empty gives NaN and sets bit 0 of *err_flag (torch raises there).  occupied_out (optional): (n, 2) int32
 * voxel counts.  n <= 65535 per call. */
size_t nm_voxel_chamfer_workspace_bytes(int n, int G);
int nm_voxel_chamfer(const float* gt, float* recon, int n, int G, int binarize_recon, float* out, int* occupied_out,
                     int* err_flag, void* workspace, void* stream);
/* utils/eval_utils.py:60-90 `semantic_scores`: rows of keypoints (F, K, 4) with intensity < threshold are
 * overwritten IN PLACE by (1e4, 1e4, 1e4, 1) (:68-69); idx_out (F, Kgt) int64 = nearest detected keypoint of
 * every ground-truth joint gt_keypoints (F, Kgt, 3); hist (Kgt, K) int32 = its histogram over the F frames. */
int nm_semantic_nearest(float* keypoints, const float* gt_keypoints, int F, int K, int Kgt, float threshold,
                        long long* idx_out, int* hist, void* stream);
/* vis_retarget.py:21-62 `extract_skin_weights`: points (N, 3), keypoints (K, 4), parents (K) int32, root =
 * priority.indices[0]; skin_out (N, K) fp32 (two non-zeros per row); nearest_out (optional, N) int32 = the chosen
 * bone; bit 0 of *err_flag is set when the parent walk over invalid joints does not terminate. */
int nm_skin_weights(const float* points, int N, const float* keypoints, const int* parents, int K, int root,
                    float hardness, float threshold, float* skin_out, int* nearest_out, int* err_flag, void* stream);
/* vis_retarget.py:279-287,:300: forward kinematics of the retargeted skeleton.  R (T, K, 3, 3), offset (K, 3),
 * root_pos (T, 3), order = priority.indices, parents (K) int32 -> pos_out (T, K, 3), clipped to [-1, 1] if clip. */
int nm_retarget_fk(const float* R, const float* offset, const float* root_pos, const int* order, const int* parents,
                   int T, int K, int clip, float* pos_out, void* stream);
/* vis_retarget.py:263-270,:315-322: linear blend skinning.  points (N, 3), joints (K, 3), R_inv (K, 3, 3) or NULL
 * (identity), T3x4 (T, K, 3, 4) = [R | pos], skin (N, K) -> out (T, N, 3). */
int nm_linear_blend_skinning(const float* points, int N, const float* joints, const float* R_inv, const float* T3x4,
                             const float* skin, int T, int K, float* out, void* stream);

/* ---- config #4 training step: backward kernels (DESIGN.md §7) -----------------------------------------
 * Weight gradient of a stride-1 3x3x3 "same" Conv3d (what autograd computes for vox_modules.py:8-47 /
 * kypt_detector.py:417-460 layers): x act (n, D, H, W, Cin), grad_out act (n, D, H, W, Cout) ->
 * dw (Cout, Cin, 3, 3, 3) fp32 in the nn.Conv3d weight layout, fully overwritten, multiplied by out_scale.  Cin, Cout multiples of 32 (<= 256),
 * W in {16, 32, 48, 64}.  First version on mma.sync with a fixed-order split-K reduction (bit-reproducible).
 * (The data gradient needs no entry point of its own: it is nm_conv3d_tc with flipped, transposed weights.) */
size_t nm_conv3d_k3_wgrad_workspace_bytes(int n, int D, int H, int W, int Cin, int Cout);
int nm_conv3d_k3_wgrad(const void* x, const void* grad_out, int n, int D, int H, int W, int Cin, int Cout,
                       float out_scale, float* dw, void* workspace, void* stream);
/* The same weight gradient on the 5th-gen tensor cores: tcgen05.mma with MN-major operands straight from the TMA-loaded
 * voxel-major tiles (K = voxels), kw shifts stacked along M and the three kh rows along N through the descriptor
 * strides, fp32 accumulators in TMEM, fixed-order split-K (bit-reproducible).  Cin, Cout multiples of 32 (<= 256),
 * W in {16, 32, 64, 128}, H a multiple of 256 / W: nm_conv3d_k3_wgrad_tc_supported. */
int nm_conv3d_k3_wgrad_tc_supported(int n, int D, int H, int W, int Cin, int Cout);
size_t nm_conv3d_k3_wgrad_tc_workspace_bytes(int n, int D, int H, int W, int Cin, int Cout);
int nm_conv3d_k3_wgrad_tc(const void* x, const void* grad_out, int n, int D, int H, int W, int Cin, int Cout,
                          float out_scale, float* dw, void* workspace, void* stream);
/* Backward of z = LeakyReLU_0.01(GroupNorm(x)) (leaky != 0) or of GroupNorm alone (modules/vox_modules.py:8-75 under
 * autograd): x, grad_out (= dL/dz), grad_in (= dL/dx) act (n, S, C) fp16; gamma, beta (C) fp32.  Optional fp32 outputs,
 * summed over the n samples and multiplied by out_scale (= 1 / loss scale): dgamma, dbeta (C) and dxsum (C) = the sum of
 * grad_in over samples and voxels, i.e. the gradient of the bias of the convolution that produced x.  Streaming kernels
 * for C in {8, 16, 32, 64, 128, 256} with 8 | channels per group; any other (C, groups) (the hour-glass's 48 / 72
 * channels) on small tensors.  mean_rstd (n, groups, 2) + xsum (n, C) kept from the forward (nm_groupnorm_finalize)
 * skip the statistics pass; when null they are recomputed from x.  Fixed-order reductions (bit-reproducible). */
size_t nm_groupnorm_backward_workspace_bytes(int n, int C, int groups);
int nm_groupnorm_backward(const void* x, const void* grad_out, const float* gamma, const float* beta, int n, long long S,
                          int C, int groups, float eps, int leaky, float out_scale, const float* mean_rstd,
                          const float* xsum, void* grad_in, float* dgamma, float* dbeta, float* dxsum, void* workspace,
                          void* stream);

/* Weight gradient of the convolutions the slab kernel above does not cover - 1x1, k2/s2 "pool", ConvTranspose3d(k2, s2),
 * k3 on small grids or with 48 / 72 channels (modules/vox_modules.py:12-68 under autograd):
 *   dw[a][b][tap] = out_scale * sum_u small_side[u][a] * large_side[u * stride + tap - pad][b]
 * nn.Conv3d: small_side = dL/dy (n, Ds, Hs, Ws, Cout), large_side = x -> dw (Cout, Cin, k, k, k);
 * nn.ConvTranspose3d: small_side = x (n, Ds, Hs, Ws, Cin), large_side = dL/dy -> dw (Cin, Cout, 2, 2, 2).
 * (k, stride) in {(1, 1), (3, 1), (2, 2)}; channels multiples of 8, <= 256.  mma.sync, fixed-order split-K. */
size_t nm_conv3d_wgrad_gather_workspace_bytes(int n, int Ds, int Hs, int Ws, int Ca, int Cb, int k, int stride);
int nm_conv3d_wgrad_gather(const void* small_side, const void* large_side, int n, int Ds, int Hs, int Ws, int Ca, int Cb,
                           int k, int stride, float out_scale, float* dw, void* workspace, void* stream);

/* Data gradient of the k2/s2 "pool" convs (modules/vox_modules.py:53 under autograd) on the tensor cores: the transposed
 * conv is a 1x1 conv dL/dy -> (tap, ci) (nm_conv3d_tc with the weight read as [(tap, ci)][co]) followed by this scatter
 * of the tap-major result y (n, D, H, W, ntaps, C) - taps tap0 .. tap0 + ntaps - 1, tap = kd*4 + kh*2 + kw - to
 * out (n, 2D, 2H, 2W, C). */
int nm_depth_to_space2(const void* y, void* out, int n, int D, int H, int W, int C, int tap0, int ntaps, void* stream);

/* Backward of nm_upsample2x without the fused prologue (nn.Upsample(scale 2, trilinear, align_corners=False),
 * model/kypt_detector.py:427,441): grad_out act (n, 2D, 2H, 2W, C) -> grad_in act (n, D, H, W, C); three separable
 * passes (w, h, d) through two fp16 intermediates in `workspace`. */
size_t nm_upsample2x_backward_workspace_bytes(int n, int D, int H, int W, int C);
int nm_upsample2x_backward(const void* grad_out, void* grad_in, int n, int D, int H, int W, int C, void* workspace,
                           void* stream);

/* Backward of nm_final_recon with the BCE (model/kypt_detector.py:410,453-457,:91-92).  x, a, b, w, bias, first_frame,
 * recon (the saved forward output), target as in the forward; grad_bce (n) = dL/d(per-frame BCE mean).
 * grad_act act (n, S, C) = grad_scale * dL/d(LeakyReLU(x*a+b)) (feed it to nm_groupnorm_backward with x);
 * dw (C), dbias (1) fp32 = gradient of the 1x1 conv (not scaled). */
size_t nm_final_recon_backward_workspace_bytes(int n);
int nm_final_recon_backward(const void* x, const float* a, const float* b, const float* w, float bias, const float* bias_dev,
                            const float* first_frame, int frames_per_clip, float sharpness, float translation,
                            const float* recon, const float* target, const float* grad_bce, float grad_scale,
                            void* grad_act, float* dw, float* dbias, void* workspace, int n, int S, int C, void* stream);

/* The same backward fused with the GroupNorm + LeakyReLU that feeds the tail (decode_voxel_from_combined_representation
 * .12 - .14): the tail's gradient w.r.t. the activated tensor is rank one per voxel (w[c] * dx14[v]) and is never
 * written.  gamma / beta / groups: that GroupNorm; mean_rstd (n, groups, 2), xsum (n, C): its forward statistics
 * (nm_groupnorm_finalize).  Outputs: grad_x act (n, S, C) = grad_scale * dL/d(raw conv output), dw (C), dbias (1) of the
 * 1x1 conv, dgamma / dbeta (C) and dxsum (C) = the producing conv's bias gradient (fp32, true scale). */
size_t nm_final_recon_backward_fused_workspace_bytes(int n, long long S, int C, int groups);
int nm_final_recon_backward_fused(const void* x, const float* a, const float* b, const float* w, float bias,
                                  const float* bias_dev, float sharpness,
                                  const float* recon, const float* target, const float* grad_bce, float grad_scale,
                                  const float* gamma, const float* beta, const float* mean_rstd, const float* xsum,
                                  int groups, void* grad_x, float* dw, float* dbias, float* dgamma, float* dbeta,
                                  float* dxsum, void* workspace, int n, long long S, int C, void* stream);

/* Backward of nm_heatmap_head (model/kypt_detector.py:273-297,336-343; utils/kypt_detector_utils.py:28-55).
 * mode 1: inputs as the forward plus its saved outputs heat, keypoints, heat_mean; upstream gradients (each optional)
 *   grad_keypoints (n, K, 4), grad_heat_mean (n, K), grad_heat (n, K, g^3).  Outputs: grad_feature act (n, g^3, C) times
 *   grad_scale; dq_out (n, K, g^3) = dL/d(pre-Softplus map) (input of the mode-0 call); dw1 (K, C), db1 (K),
 *   dprop (3) = gradient of the propagate conv (w0, w1, bias).
 * mode 0 (spatio-temporal head, n = clips): upstream = pw1 * sum over the clip's frames of dq_in ((n*frames_per_clip, K,
 *   g^3)) [+ grad_heat]; outputs grad_feature, dw1, db1. */
size_t nm_heatmap_head_backward_workspace_bytes(int n, int C, int K);
int nm_heatmap_head_backward(const void* feature, const float* w1, const float* b1, int n, int g, int C, int K, int mode,
                             const float* prev, int frames_per_clip, float pw0, float pw1, float pb, const float* prop_dev,
                             const float* linspace, const float* heat, const float* keypoints, const float* heat_mean,
                             const float* grad_keypoints, const float* grad_heat_mean, const float* grad_heat,
                             const float* dq_in, float grad_scale, void* grad_feature, float* dq_out, float* dw1,
                             float* db1, float* dprop, void* workspace, void* stream);

/* Backward of nm_decoder_adjust in keypoint mode (model/kypt_detector.py:381,404-408 + the Gaussian render,
 * utils/kypt_detector_utils.py:57-90).  grad_out, out: act (n, g^3, 128) (out = the saved forward output; grad_out carries
 * grad_scale).  Outputs: grad_first_feature act (n_clips, g^3, 128) times grad_scale; grad_keypoints (n, K, 4) fp32
 * (through gauss_t of every frame and gauss_0 of the clip's first frame); dweight (128, 2K+131), dbias (128) fp32. */
size_t nm_decoder_adjust_backward_workspace_bytes(int n_clips, int frames_per_clip);
int nm_decoder_adjust_backward(const void* grad_out, const void* out, const void* first_feature, const float* keypoints,
                               const float* weight, int n_clips, int frames_per_clip, int g, int K, const float* linspace,
                               float gauss_width, float grad_scale, void* grad_first_feature, float* grad_keypoints,
                               float* dweight, float* dbias, void* workspace, void* stream);

/* Backward of nm_chamfer_vol_fit (utils/kypt_detector_utils.py:141-157): grad_out (n) -> grad_keypoints (n, K, 4). */
size_t nm_chamfer_vol_fit_backward_workspace_bytes(int n, int K);
int nm_chamfer_vol_fit_backward(const float* seq, const float* keypoints, const float* linspace, const float* grad_out,
                                int n, int K, int G, float* grad_keypoints, void* workspace, void* stream);

/* Weight gradient of the CoordConv first layer (add_coord_channels + Conv3d(4, Cout, k5, pad 2),
 * utils/kypt_detector_utils.py:4-26, model/kypt_detector.py:266): occ (n, G, G, G) fp32 (any values: the
 * spatio-temporal branch feeds the frame mean), grad_out act (n, G, G, G, Cout) -> dw (Cout, 4, 5, 5, 5) fp32 times
 * out_scale.  The coordinate channels are never materialised: their sums follow from 125 positional bins of the
 * moments of grad_out; the occupancy channel is a gather over the non-zero voxels. */
size_t nm_first_conv_wgrad_workspace_bytes(int n, int Cout);
int nm_first_conv_wgrad(const float* occ, const void* grad_out, const float* linspace, int n, int G, int Cout,
                        float out_scale, float* dw, void* workspace, void* stream);

/* Optimizer of the training loop (train.py:380-409: torch.optim.Adam(lr) with default betas / eps, no weight decay) as
 * one launch over a flat parameter buffer.  grad is multiplied by grad_mul first (unscaling / averaging); when
 * *skip_flag != 0 (set by nm_grad_nonfinite: some gradient is inf / NaN) the step leaves everything untouched. */
int nm_grad_nonfinite(const float* grad, long long count, int* flag, void* stream);
int nm_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long count, float lr, float beta1,
                 float beta2, float eps, int step, float grad_mul, const int* skip_flag, void* stream);
/* The same step with the step count on the device: counters[0] = steps applied so far (the bias corrections use
 * counters[0] + 1), counters[1] = steps skipped; both are advanced by the call.  No argument depends on host-side training
 * state, so a CUDA graph that captured a whole training step (forward, backward, nm_grad_nonfinite, this call) can be
 * replayed. */
int nm_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long count, float lr, float beta1,
                     float beta2, float eps, int* counters, float grad_mul, const int* skip_flag, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NM_B200_H */
