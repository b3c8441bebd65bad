/* lfb200.h — C ABI of the B200-native LatentFusion reconstruct->render hot path.
 *
 * The reference (NVlabs/latentfusion) is pure Python/PyTorch and has no FFI of its own
 * (SURVEY.md §8b); the boundary a maintainer binds is therefore the set of ATen ops its hot path
 * dispatches to.  Each entry point below names the reference call site it replaces
 * (paths relative to /root/reference/latentfusion/).  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - plain C: pointers + sizes only, no torch types; every pointer is a DEVICE pointer unless it
 *     says "host"; the caller owns every buffer (the library never allocates or frees, never keeps
 *     a pointer past the call, never synchronises) so every call is CUDA-graph capturable.
 *   - `stream` is a cudaStream_t passed as void*.
 *   - feature maps are dense channels-last fp32: 3-D [N][D][H][W][C], 2-D [N][H][W][C].
 *   - return value: 0 ok; <0 invalid argument (lf_last_error() has the text); >0 a cudaError_t.
 *   - thread safety: no global mutable state on the product path besides the thread-local last-error string.
 *     Development only: the option table (environment, read once; lf_set_option) and a diagnostic timeline
 *     buffer that a kernel writes only when LFB200_TC_DEBUG & 8 is set.
 */
#ifndef LFB200_H
#define LFB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LF_OK 0
#define LF_EINVAL (-1)
#define LF_EUNSUPPORTED (-2)

/* Per-camera constant block consumed by the resamplers (floats). */
#define LF_CAM_STRIDE 40
/* object->camera layout (geometry.py:469-531, :669-685):
 *   [0..11]  cam_to_obj rows 0..2 (3x4, row major)      geometry.py:211-213
 *   [12..15] viewport x0, y0, width, height             geometry.py:169-175
 *   [16..19] u0, v0, fu, fv                             geometry.py:183-197
 *   [20] znear  [21] z_span  [22] 2/cube_size           geometry.py:249-251, :491, :684
 * camera->object layout (geometry.py:599-654):
 *   [0..11]  obj_to_cam rows 0..2                       geometry.py:207-209
 *   [12..15] viewport x0, y0, width, height
 *   [16..27] intrinsic 3x4                              geometry.py:636
 *   [28] znear  [29] zfar  [30] cube_size */
/* Gradient block produced by lf_resample_o2c_bwd_cam: [0..15] = d/d(cam[0..15]), [16] = d/d(znear). */
#define LF_CAMGRAD_STRIDE 20

const char* lf_version(void);
const char* lf_last_error(void);
/* Number of SMs of the current device (used by callers to size workspaces). */
int lf_sm_count(void);
/* Tuning / A-B switches are the LFB200_* environment variables, read ONCE at first use (never per launch);
 * lf_set_option overrides one by name afterwards (tests and profiling tools; not thread-safe).  The kernels' mbarrier
 * waits are bounded: a pipeline bug prints "lfb200: mbarrier wait timed out" and traps (the launch then reports a CUDA
 * error) instead of hanging the device. */
int lf_set_option(const char* name, int value);

/* ---- K1: ObjectToCameraTransform.forward  (modules/geometry.py:669-690; F.grid_sample :17) ----
 * vol  [B][S][S][S][C]   one latent cube per object (NOT replicated per camera; models.py:493-494)
 * cam  [N][LF_CAM_STRIDE]; camera n samples object n / (N/B)
 * out  [N][S][S][S][C] */
int lf_resample_o2c_fwd(const float* vol, const float* cam, float* out,
                        int B, int N, int C, int S, void* stream);
/* The same resample written straight into the split-planar activation layout of lf_split_pack (out_split:
 * lf_split_bytes(N, S, S, S, C) bytes, zero halo included) for a following lf_conv3d_dz: no dense fp32 copy of the
 * [N][S^3][C] volumes and no packing pass.  C in {16, 32, 64} (lf_resample_o2c_fwd_split_supported). */
int lf_resample_o2c_fwd_split_supported(int C, int S);
int lf_resample_o2c_fwd_split(const float* vol, const float* cam, void* out_split,
                              int B, int N, int C, int S, void* stream);
/* backward w.r.t. the camera block (the pose loop's gradient; replaces grid_sampler_3d_backward's
 * grad_grid + the autograd of geometry.py:469-531,:669-685).
 * grad_cam [N][LF_CAMGRAD_STRIDE]; workspace: lf_resample_o2c_bwd_cam_ws(N,S) floats. */
int64_t lf_resample_o2c_bwd_cam_ws(int N, int S);
int lf_resample_o2c_bwd_cam(const float* grad_out, const float* vol, const float* cam,
                            float* grad_cam, float* workspace,
                            int B, int N, int C, int S, void* stream);
/* the same gradient laid out as a camera block [N][LF_CAM_STRIDE] (terms 0..15 in place, d/d(znear) at [20], zeros
 * elsewhere): what lf_camera_o2c_bwd consumes, without a re-layout pass in between */
int lf_resample_o2c_bwd_cam_block(const float* grad_out, const float* vol, const float* cam,
                                  float* grad_block, float* workspace,
                                  int B, int N, int C, int S, void* stream);
/* backward w.r.t. the volume (training). grad_vol [B][S^3][C] must be zeroed by the caller. */
int lf_resample_o2c_bwd_vol(const float* grad_out, const float* cam, float* grad_vol,
                            int B, int N, int C, int S, void* stream);

/* ---- K2: CameraToObjectTransform.forward  (modules/geometry.py:625-657) ----
 * vol [V][S][S][S][C] camera-frustum volumes, out [V][S][S][S][C] object cubes. */
int lf_resample_c2o_fwd(const float* vol, const float* cam, float* out,
                        int V, int C, int S, void* stream);
int lf_resample_c2o_bwd_vol(const float* grad_out, const float* cam, float* grad_vol,
                            int V, int C, int S, void* stream);

/* ---- K3/K5/K6: Equalized conv + fused epilogue  (modules/equalized.py:57-64, blocks.py:152-164,
 *      modules/__init__.py:14-15, geometry.py:704-749) ----
 * One implicit-GEMM entry point covers every convolution on the path:
 *   ndim=3, k=3|1 : EqualizedConv3d          (camera/object blocks, GRU gates, OutputBlock3d)
 *   ndim=2, k=3|1 : EqualizedConv2d          (UNet2d blocks, InputBlock, heads, 2D->3D lift)
 *   ndim=1        : "depth-collapse" GEMM of FactorProjection3d2d: x [N][S][H][W][C] -> y [N][H][W][Cout],
 *                   S taps along depth (geometry.py:744-749); w packed [S][Cin][Cout]
 *   ndim=-1       : "depth-expand" GEMM of FactorProjection2d3d: x [N][H][W][Cin] -> y [N][S][H][W][Cout],
 *                   one 1x1 GEMM per depth slice (geometry.py:724-728); w packed [S][Cin][Cout], bias [S][Cout];
 *                   PixelNorm then runs over the whole (S x Cout) group of a pixel, as the reference
 *                   normalises before its view(); rnorm is [N*H*W].
 * x   [N][(D)][H][W][Cin]; w packed [taps][Cin][Cout] (host repack of [Cout][Cin][k..]); bias [Cout]
 * y = conv(x,w)*scale + bias ; act: 0 none, 1 LeakyReLU(slope) ; norm: 0 none, 1 PixelNorm over Cout
 * y   [N][(D)][H][W][Cout]; rnorm (nullable) [positions] = sqrt(mean_c(a^2)+1e-8) saved for backward. */
typedef struct {
    int ndim;          /* 2 or 3: regular conv; 1: depth-collapse; -1: depth-expand (see above) */
    int n, d, h, w;    /* input extent (d = 1 for 2-D) */
    int cin, cout;
    int k;             /* kernel size (1 or 3; for ndim==1: number of depth taps = d) */
    float scale;       /* He constant sqrt(2/fan_in) */
    int act;           /* 0 none, 1 leaky relu */
    float slope;
    int norm;          /* 0 none, 1 pixel norm */
    int precision;     /* 0 = fp32 CUDA-core path (exact), 1 = tcgen05 bf16x3 split, 2 = tcgen05 bf16 */
} lf_conv_desc;

int lf_conv_fwd(const lf_conv_desc* desc, const float* x, const float* w, const float* bias,
                float* y, float* rnorm, void* stream);
/* ---- depth-batched tcgen05 3x3x3 convolution on split-planar activations (csrc/conv3d_dz.cu) ----
 * Same reference op as lf_conv_fwd with ndim = 3, k = 3 (modules/equalized.py:57-64 + blocks.py:152-158), for
 * Cout <= 32 (Cout % 4 == 0), precision 1 (bf16x3 in ONE pass) or 2 (bf16).  Activations travel between
 * convolutions in the library's internal "split-planar" layout
 *     [part: hi | lo][N][D][C_pad/8][H+2][W+2][8] bf16      (x ~ hi + lo; zero halo; C_pad = C rounded up to 16)
 * which a kernel stages with 1-D bulk TMA copies (cp.async.bulk).  lf_split_bytes gives the buffer size in bytes,
 * lf_split_pack converts a dense channels-last fp32 tensor [N][D][H][W][C] into it (halo and padding channels zeroed).
 * lf_conv3d_dz reads x_split and writes y32 (fp32 channels-last [N][D][H][W][Cout], nullable) and/or y_split
 * (split-planar with Cout channels, nullable; the kernel writes its whole halo) and rnorm (nullable).
 * `w_packed` comes from lf_conv3d_dz_pack_weights applied to the [27][Cin][Cout] fp32 pack (tap = (dz*3+dy)*3+dx).
 * Error contract of every tcgen05 kernel: all mbarrier waits are bounded; a pipeline fault prints one line and
 * traps (cudaErrorLaunchFailure at the next synchronisation) instead of hanging the device. */
int lf_conv3d_dz_supported(const lf_conv_desc* desc);
int64_t lf_split_bytes(int n, int d, int h, int w, int c);
int lf_split_pack(const float* x, void* out_split, int n, int d, int h, int w, int c, void* stream);
int64_t lf_conv3d_dz_weight_bytes(int cin, int cout);
int lf_conv3d_dz_pack_weights(const float* w27, void* out, int cin, int cout, void* stream);
int lf_conv3d_dz(const lf_conv_desc* desc, const void* x_split, const void* w_packed, const float* bias,
                 float* y32, void* y_split, float* rnorm, void* stream);
/* bwd-data (desc: cin = forward Cout, cout = forward Cin, act = norm = 0) with the PixelNorm/LeakyReLU backward of the
 * layer that produced the forward input fused into the epilogue (replaces lf_actnorm_bwd of that layer: its output
 * y_prev arrives in split-planar form, rnorm_prev are its saved norms); writes du_prev dense and/or split-planar. */
int lf_conv3d_dz_bwd_epi(const lf_conv_desc* desc, const void* du_split, const void* w_packed,
                         const void* y_prev_split, const float* rnorm_prev, int prev_act, float prev_slope,
                         int prev_norm, float* du_prev32, void* du_prev_split, void* stream);
/* lf_actnorm_bwd for a 3-D layer with C in {16, 32} that writes du in split-planar form (du_split, with its zero halo)
 * for the layer's bwd-data convolution, and dense fp32 too when `du` is non-null. */
int lf_actnorm_bwd_split(const float* gy, const float* y, const float* rnorm, float* du, void* du_split,
                         int n, int d, int h, int w, int c, int act, float slope, int norm, void* stream);
/* diagnostic: same launch, plus SM-clock stamps of CTA 0's pipeline roles in `stamps` (device, 4*64*2 int64) */
int lf_conv3d_dz_timeline(const lf_conv_desc* desc, const void* x_split, const void* w_packed, const float* bias,
                          float* y32, void* y_split, float* rnorm, void* stamps, void* stream);

/* tcgen05 path (precision 1|2): `w` passed to lf_conv_fwd must point to weights pre-packed by
 * lf_conv_tc_pack_weights (bf16 hi part followed by the bf16 lo part, UMMA no-swizzle K-major layout
 * [part][tap][Cin_pad/8][Cout_pad][8]); lf_conv_tc_weight_bytes gives the buffer size.  Shapes the
 * tensor-core kernel does not cover (lf_conv_tc_supported == 0, e.g. Cin % 4 != 0, depth-collapse/expand)
 * must be run with precision 0. */
int64_t lf_conv_tc_weight_bytes(int taps, int cin, int cout);
int lf_conv_tc_pack_weights(const float* w_packed /* [taps][Cin][Cout] fp32 */, void* out,
                            int taps, int cin, int cout, void* stream);
int lf_conv_tc_supported(const lf_conv_desc* desc);
/* kernel launches of lf_conv_fwd on the tcgen05 path for this descriptor: 1 (bf16, and bf16x3 of 2-D layers whose hi and
 * lo slabs fit side by side: the one-pass form), 2|3 (bf16x3 otherwise); 0 = not covered */
int lf_conv_tc_passes(const lf_conv_desc* desc);
/* Backward-data of a Block conv with the PixelNorm/LeakyReLU backward (lf_actnorm_bwd) fused into the operand
 * staging of the tcgen05 kernel: gx = conv_T(du) * scale with du = LeakyReLU'(y) * PixelNorm^T(gy) never written
 * to HBM.  `desc` describes the backward conv (cin = forward Cout, cout = forward Cin, act = norm = 0);
 * fwd_* are the forward layer's epilogue flags; y_fwd / rnorm_fwd its saved output and norm.  Returns
 * LF_EUNSUPPORTED for shapes outside the kernel's coverage (caller then runs lf_actnorm_bwd + lf_conv_fwd). */
int lf_conv_bwd_data_fused(const lf_conv_desc* desc, const float* gy, const float* y_fwd, const float* rnorm_fwd,
                           int fwd_act, float fwd_slope, int fwd_norm, const float* w_tc_packed, float* gx,
                           void* stream);

/* du = d(loss)/d(pre-activation conv output incl. scale&bias) from gy, y (post-norm output), rnorm.
 * PixelNorm + LeakyReLU backward fused.  Elements are y[(o*gd + t)*inner + p][c]; one norm group =
 * all (t, c) of a fixed (o, p): gd = 1 for ordinary convs (outer = positions, inner = 1); for the
 * depth-expand lift outer = N, gd = S, inner = H*W. */
int lf_actnorm_bwd(const float* gy, const float* y, const float* rnorm, float* du,
                   int64_t outer, int gd, int64_t inner, int c, int act, float slope, int norm, void* stream);
/* dx = conv_transpose(du * scale, w): call lf_conv_fwd with the flipped/transposed packed weights
 * (host repack) and act=norm=0.  Weight / bias gradients (training): */
int lf_conv_bwd_weight(const lf_conv_desc* desc, const float* x, const float* du,
                       float* grad_w_packed /* [taps][Cin][Cout], zeroed by caller */,
                       float* grad_bias /* [Cout], zeroed by caller */, void* stream);

/* ---- Interpolate (modules/__init__.py:18-33): mode 0 nearest, 1 (bi/tri)linear align_corners=False;
 *      factor 2 (up) or -2 (down by 2).  x [N][(D)][H][W][C]. */
int lf_interp_fwd(const float* x, float* y, int ndim, int n, int d, int h, int w, int c,
                  int mode, int factor, void* stream);
int lf_interp_bwd(const float* gy, float* gx, int ndim, int n, int d, int h, int w, int c,
                  int mode, int factor, void* stream);

/* ---- K4: view-axis fusion (recon/fusion.py:45-57; functional.py:47-49) ----
 * z [B][V][P][C] -> out [B][P][C]; kind 0 max, 1 mean, 2 abs_max, 3 median (lower median, as torch). */
int lf_fuse_pool_fwd(const float* z, float* out, int B, int V, int64_t P, int C, int kind, void* stream);
int lf_fuse_pool_bwd(const float* gout, const float* z, float* gz, int B, int V, int64_t P, int C,
                     int kind, void* stream);
/* ConvGRUCell gate math (modules/gru.py:36-43), conv outputs already computed:
 *   stage 1: update = sigmoid(u_pre), reset = sigmoid(r_pre), hr = h * reset
 *   stage 2: h_new = h*(1-update) + o*update */
int lf_gru_gates1(const float* u_pre, const float* r_pre, const float* h, float* update, float* hr,
                  int64_t numel, void* stream);
int lf_gru_gates2(const float* h, const float* update, const float* o, float* h_new,
                  int64_t numel, void* stream);
/* backward of the two gate kernels (autograd of modules/gru.py:38-41), one pass each */
int lf_gru_gates1_bwd(const float* g_update, const float* g_hr, const float* update, const float* r_pre, const float* h,
                      float* g_u_pre, float* g_r_pre, float* g_h, int64_t numel, void* stream);
int lf_gru_gates2_bwd(const float* g, const float* h, const float* update, const float* o, float* g_h, float* g_update,
                      float* g_o, int64_t numel, void* stream);
/* ConvLSTM gate non-linearities (modules/lstm.py:41-56): gates [P][4*hidden] channels-last = (i | f | o | g)
 * pre-activations; c_next = sig(f) c_cur + sig(i) tanh(g); h_next = sig(o) tanh(c_next).  bwd: g_h / g_c nullable. */
int lf_lstm_gates_fwd(const float* gates, const float* c_cur, float* h_next, float* c_next, int64_t positions, int hidden,
                      void* stream);
int lf_lstm_gates_bwd(const float* g_h, const float* g_c, const float* gates, const float* c_cur, float* g_gates,
                      float* g_c_cur, int64_t positions, int hidden, void* stream);
/* softmax over the outer axis V of scores [B][V][P] and the weighted sum of z [B][V][P][C] over it, channels-last:
 * the BlendFuser's view blend (recon/fusion.py:92-96).  Writes the weights [B][V][P] too.  bwd: g_weights and g_z nullable. */
int lf_softmax_blend_fwd(const float* scores, const float* z, float* weights, float* out, int b, int v, int64_t p, int c,
                         void* stream);
int lf_softmax_blend_bwd(const float* g_out, const float* g_weights, const float* weights, const float* z, float* g_scores,
                         float* g_z, int b, int v, int64_t p, int c, void* stream);
/* projection_type='sum' (recon/models.py:436-437): x [N][D][HW][C] -> out [N][HW][C] */
int lf_depth_sum_fwd(const float* x, float* out, int n, int d, int64_t hw, int c, void* stream);

/* ---- camera algebra (modules/geometry.py:106-108,147-163,207-213,249-255; three/quaternion.py:287-311,39-93) ----
 * The ten learnable floats of each hypothesis -> the object->camera constant block, and its analytic VJP
 * (grad_block: only entries [0..15] and [20] are read). */
int lf_camera_o2c_fwd(const float* log_quaternion /*[n][3]*/, const float* translation /*[n][3]*/,
                      const float* viewport /*[n][4]*/, const float* intrinsic /*[n][12]*/,
                      float* block /*[n][LF_CAM_STRIDE]*/, int n, float z_span, float cube_size, void* stream);
int lf_camera_o2c_bwd(const float* log_quaternion, const float* translation, const float* grad_block,
                      float* grad_log_quaternion, float* grad_translation, float* grad_viewport, int n, void* stream);
/* Batched per-hypothesis optimiser (pose/estimation.py:582-594,664-666): torch.optim.Adam single-tensor maths with
 * a per-row learning rate over param [n][width]; ReduceLROnPlateau(mode min, rel threshold, cooldown 0) per row. */
int lf_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int n, int width,
                 const float* step_count /*[1], already incremented*/, const float* lr /*[n]*/,
                 float beta1, float beta2, float eps, void* stream);
int lf_plateau_step(const float* rank_loss /*[n]*/, float* lr, float* best, float* num_bad, int n,
                    float threshold, float patience, float factor, void* stream);
/* Loss combination + bookkeeping of one refinement iteration (pose/estimation.py:611-660; replaces ~35 elementwise
 * launches of the autograd graph of sum(w*term).mean() and of the history snapshots): rank[i] = sum_k w_rank[k]*terms[i][k]
 * and the same with w_opt (left to right), grad_terms[i][k] = w_opt[k] / n (the gradient optim.mean().backward() hands
 * lf_pose_loss_bwd), and the snapshot of (rank, optim, terms, log_quaternion, translation) into the chunk history
 * h_rank/h_optim [chunk][n], h_terms [chunk][k][n], h_lq/h_tr [chunk][n][3] at *slot, which then advances modulo chunk;
 * *step_count += 1 when given (the batched Adam's step counter). */
int lf_refine_record(const float* terms /*[n][k]*/, int n, int k, const float* w_rank /*[k]*/, const float* w_opt /*[k]*/,
                     const float* log_quaternion /*[n][3]*/, const float* translation /*[n][3]*/, float* rank /*[n]*/,
                     float* grad_terms /*[n][k]*/, float* h_rank, float* h_optim, float* h_terms, float* h_lq, float* h_tr,
                     long long* slot /*[1]*/, int chunk, float* step_count /*[1], nullable*/, void* stream);

/* ---- fused pose-loss head (recon/models.py:455-484 interpret_logits; modules/geometry.py:261-285 uncrop,
 *      :555-558 denormalize_depth; pose/estimation.py:70-118 default_pose_loss; pose/utils.py:81-117) ----
 * depth_logits, mask_logits [N][P][P] (the two heads of the Photographer); viewport [N][4] (x0,y0,x1,y1);
 * tz [N] camera translation z; target_depth / target_mask [height][width] (one target observation).
 * terms [N][4] = ov_depth, depth, iou, mask.  sums [N][8] is scratch carried from fwd to bwd.  workspace is device
 * scratch of lf_pose_loss_fwd_ws / lf_pose_loss_bwd_ws bytes: every reduction adds per-block or per-pixel partials in
 * a fixed order (no atomics), so the same inputs give the same bits on every run. */
typedef struct {
    int n, p;              /* hypotheses, crop side */
    int width, height;     /* full frame */
    float z_span, eps;     /* Camera.z_span; denormalize_depth eps (0.01) */
    /* layout of the logit maps and of tz, in floats; 0 = dense ([N][P][P] maps, tz[N]).  The decoder's fused heads write
     * channels-last logits [N][P][P][H]: depth_logits = base, mask_logits = base + 1, pix_stride = H, hyp_stride = P*P*H;
     * tz = translation + 2 with tz_stride = 3.  The gradients use the layout of their inputs; lf_pose_loss_bwd writes
     * every element of the two logit maps, of grad_viewport and the N entries of grad_tz, and nothing in between. */
    int pix_stride, hyp_stride, tz_stride;
} lf_loss_desc;
int lf_pose_loss_fwd(const lf_loss_desc* desc, const float* depth_logits, const float* mask_logits,
                     const float* viewport, const float* tz, const float* target_depth, const float* target_mask,
                     float* sums, float* terms, void* workspace, void* stream);
int64_t lf_pose_loss_fwd_ws(const lf_loss_desc* desc);   /* bytes of workspace for lf_pose_loss_fwd / _search_fwd */
int64_t lf_pose_loss_bwd_ws(const lf_loss_desc* desc);   /* bytes of workspace for lf_pose_loss_bwd */
/* forward-only variant for the coarse search (CrossEntropyPoseEstimator: estimation.py:187-197 multiplies the crop's
 * metric depth by the crop's sigmoid(mask) before the loss pastes it into the frame); same outputs as lf_pose_loss_fwd */
int lf_pose_loss_search_fwd(const lf_loss_desc* desc, const float* depth_logits, const float* mask_logits,
                            const float* viewport, const float* tz, const float* target_depth,
                            const float* target_mask, float* sums, float* terms, void* workspace, void* stream);
int lf_pose_loss_bwd(const lf_loss_desc* desc, const float* depth_logits, const float* mask_logits,
                     const float* viewport, const float* tz, const float* target_depth, const float* target_mask,
                     const float* sums, const float* grad_terms /* [N][4] */,
                     float* grad_depth_logits, float* grad_mask_logits, float* grad_viewport /* [N][4] */,
                     float* grad_tz /* [N] */, void* workspace, void* stream);

/* ---- wide 3x3x3 layers: weights streamed through shared memory (csrc/conv3d_ws.cu) ----
 * The same reference op as lf_conv3d_dz for the released network widths (tools/train/train.sh:37-46: 64/128/256-channel
 * camera / object blocks on a 16^3 latent), where 27*Cin*Cout weights do not fit in shared memory: one item = (sample,
 * output plane, chunk of 64|128 output channels); the activation slab of one plane and one 32-channel input group is
 * staged by bulk TMA, weight tiles of one (dz, group, tap) stream through a 4-slot ring, accumulators of all M-tiles of
 * the (small) plane live in TMEM across the whole K loop.  x_split: split-planar input (Cin padded to 16 must be a
 * multiple of 32); y32 fp32 channels-last; PixelNorm (desc->norm) runs as a second small kernel over `scratch`
 * (lf_conv3d_ws_scratch floats) and writes rnorm.  Also takes 2-D 3x3 layers (ndim 2, d = 1: one plane per image, the
 * U-Nets' 128..512-channel maps); a plane larger than TMEM / shared memory hold at once is cut into tile groups that
 * stream the weights again (row pitch up to ~130 positions). */
int lf_conv3d_ws_supported(const lf_conv_desc* desc);
int64_t lf_conv3d_ws_weight_bytes(int taps /* 27 | 9 */, int cin, int cout);
int lf_conv3d_ws_pack_weights(const float* w_packed /* [27 | 9][Cin][Cout] */, void* out, int taps, int cin, int cout,
                              void* stream);
int64_t lf_conv3d_ws_scratch(const lf_conv_desc* desc);
int lf_conv3d_ws(const lf_conv_desc* desc, const void* x_split, const void* w_packed, const float* bias, float* y32,
                 float* rnorm, float* scratch, void* stream);

/* ---- depth collapse on the tensor cores (csrc/collapse_tc.cu) ----
 * Same reference op as lf_conv_fwd with ndim = 1 (FactorProjection3d2d + LeakyReLU + PixelNorm), reading the volume from
 * the split-planar twin its producer left (x_split) instead of the dense fp32 tensor: HBM-bound instead of FFMA-bound.
 * Cin <= 32, Cout <= 32 (multiple of 4), precision 1 | 2; y fp32 channels-last [N][H][W][Cout], rnorm nullable. */
int lf_collapse_tc_supported(const lf_conv_desc* desc);
int64_t lf_collapse_tc_weight_bytes(int depth, int cin, int cout);
int lf_collapse_tc_pack_weights(const float* w /* [depth][cin][cout] */, void* out, int depth, int cin, int cout, void* stream);
int lf_collapse_tc(const lf_conv_desc* desc, const void* x_split, const void* w_packed, const float* bias, float* y,
                   float* rnorm, void* stream);

/* ---- backward of the depth collapse fused with the producer's activation backward (csrc/expand_tc.cu) ----
 * Replaces, in the pose loop, the autograd of FactorProjection3d2d (modules/geometry.py:704-749) w.r.t. its input volume
 * followed by the PixelNorm/LeakyReLU backward of the camera block that produced it (blocks.py:152-164):
 *   du_prev = actnorm_bwd(he * du x W^T, y_prev, rnorm_prev), written in split-planar form (dense fp32 too if asked).
 * collapse_desc: the FORWARD collapse descriptor (ndim 1: cin = volume channels <= 32, cout = projected channels <= 64,
 * d = k = depth), precision 1 | 2.  du_split2d: split-planar twin of the 2-D gradient as a one-plane volume. */
int lf_expand_tc_supported(const lf_conv_desc* collapse_desc);
int64_t lf_expand_tc_weight_bytes(int depth, int cin, int cout);
int lf_expand_tc_pack_weights(const float* w /* [depth][cin][cout] */, void* out, int depth, int cin, int cout, void* stream);
int lf_expand_tc_bwd_epi(const lf_conv_desc* collapse_desc, const void* du_split2d, const void* w_packed,
                         const void* y_prev_split, const float* rnorm_prev, int prev_act, float prev_slope, int prev_norm,
                         void* du_prev_split, float* du_prev32 /* nullable */, void* stream);

/* ---- weight gradient of the 3x3x3 convolution on the tensor cores (csrc/conv3d_dw.cu) ----
 * Replaces the autograd of modules/equalized.py:57-64 w.r.t. the weight inside ReconTrainer.run_iteration
 * (tools/train/train_reconstruct.py:523-534).  x_split / du_split: split-planar volumes (layout above) of the forward
 * input and of d(loss)/d(pre-activation output).  grad_w_packed [27][Cin][Cout] = sum over positions of
 * desc->scale * x[pos + tap] (.) du[pos] (overwritten; same quantity as lf_conv_bwd_weight);
 * grad_bias [Cout] (nullable) = sum of du.  Supported: precision 1 with Cin_pad in {16, 32}, precision 2 with Cin_pad 32;
 * Cout_pad <= 32.  ws: lf_conv3d_dw_ws(desc) floats of scratch.  Deterministic (fixed-order two-stage sums). */
int lf_conv3d_dw_supported(const lf_conv_desc* desc);
int64_t lf_conv3d_dw_ws(const lf_conv_desc* desc);
int lf_conv3d_dw(const lf_conv_desc* desc, const void* x_split, const void* du_split, float* ws,
                 float* grad_w_packed, float* grad_bias, void* stream);

/* bwd-data convolution (or depth-expand, ndim -1) with the PixelNorm/LeakyReLU backward of the PRODUCER of the forward
 * input fused into the epilogue: writes du_prev = actnorm_bwd(conv_bwd_data(du), y_prev, rnorm_prev) in one kernel
 * (replaces blocks.py:152-164's autograd of conv -> LeakyReLU -> PixelNorm between two stacked convolutions).
 * `w`: tcgen05-packed weights for conv descriptors (precision 1|2), fp32 [D][Cin][Cout] for ndim -1. */
int lf_conv_bwd_data_epi_supported(const lf_conv_desc* desc);
int lf_conv_bwd_data_epi(const lf_conv_desc* desc, const float* du, const float* w, const float* y_prev,
                         const float* rnorm_prev, int prev_act, float prev_slope, int prev_norm, float* du_prev,
                         void* stream);

/* All output heads of the render decoder in one pass (recon/models.py:331-338, :448-452: several 1x1 Equalized convs
 * with 1-3 output channels each, concatenated): y[pos][h] = scale * sum_c x[pos][c] * w[h][c] + bias[h], exact fp32.
 * x [positions][C] channels-last, w [H][C], H <= 8, C = 4 * 2^k <= 128.  lf_heads_bwd: gx = scale * g . w. */
int lf_heads_fwd(const float* x, const float* w, const float* bias, float* y, int64_t positions, int c, int h,
                 float scale, void* stream);
int lf_heads_bwd(const float* g, const float* w, float* gx, int64_t positions, int c, int h, float scale, void* stream);

/* ---- IBR colour branch (SURVEY §8 f-3; forward only: the pose loop does not differentiate it) ---------------
 * IBR camera block, LF_IBR_CAM_STRIDE floats per camera:
 *   [0,12) cam_to_obj rows 0-2   [12,24) obj_to_cam rows 0-2   [24,36) obj_to_image = K * obj_to_cam (3x4)
 *   [36,40) viewport x0, y0, width, height   [40,44) u0, v0, fu, fv   [44] znear - 0.01   [45] zfar + 0.01
 * lf_ibr_reproject_fwd replaces latentfusion/ibr.py:11-93 (depth_to_warp_field + reproject_views: two batched
 * matmuls, the [Vo*Vi,H,W,2] grid, the transformed-depth image and two F.grid_sample calls, bilinear / zeros /
 * align_corners=False).  Images are planar (channel-first) like the reference's. */
#define LF_IBR_CAM_STRIDE 48
int lf_ibr_reproject_fwd(const float* image_in /* [Vi][C][H][W] */, const float* depth_in /* [Vi][H][W], used as given */,
                         const float* depth_out /* [Vo][H][W], normalised */, const float* cam_out /* [Vo][48] */,
                         const float* cam_in /* [Vi][48] */, float* image_reproj /* [Vo][Vi][C][H][W] */,
                         float* depth_reproj /* [Vo][Vi][H][W] */, int vo, int vi, int c, int h, int w, void* stream);
/* ibr.py:223-224, :231-234: out[b][c][p] = sum_i wts[b][i][per_pixel ? p : 0] * img[b][i][c][p] */
int lf_ibr_blend_fwd(const float* img /* [B][Vi][C][HW] */, const float* wts /* [B][Vi] or [B][Vi][HW] */,
                     float* out /* [B][C][HW] */, int b, int vi, int c, int hw, int per_pixel, void* stream);
/* ibr.py:237-249 warp_blend_logits: logits [B][3*Vi][H][W] = (blend | flow x | flow y); C <= 8 */
int lf_ibr_warp_blend_fwd(const float* logits, const float* image_reproj /* [B][Vi][C][H][W] */, float flow_size,
                          float* image /* [B][C][H][W] */, float* weights /* [B][Vi][H][W] */,
                          float* flow_dx /* [B][Vi][H][W] */, float* flow_dy /* [B][Vi][H][W] */,
                          int b, int vi, int c, int h, int w, void* stream);
/* Backward of the two blend heads (the IBR generator is trained through them, tools/train/train_ibr.py:367-376; the
 * reprojection itself runs without grad there).  blend: grad_wts[b][i][p] = sum_c grad_out[b][c][p] * img[b][i][c][p].
 * warp_blend: gradient of all four outputs of ibr.py:237-249 (image; blend weights / flow_dx / flow_dy upstream
 * gradients nullable) w.r.t. the logits: softmax, tanh, clamp (inclusive, as torch.clamp) and the bilinear sampler's
 * coordinate gradient (ATen grid_sampler_2d_backward, zeros padding, align_corners=False). */
int lf_ibr_blend_bwd(const float* grad_out /* [B][C][HW] */, const float* img /* [B][Vi][C][HW] */,
                     float* grad_wts /* [B][Vi][HW] */, int b, int vi, int c, int hw, void* stream);
int lf_ibr_warp_blend_bwd(const float* logits, const float* image_reproj, float flow_size, const float* grad_image,
                          const float* grad_weights, const float* grad_flow_dx, const float* grad_flow_dy,
                          float* grad_logits /* [B][3*Vi][H][W] */, int b, int vi, int c, int h, int w, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LFB200_H */
