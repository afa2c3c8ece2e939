/* mmnn_b200.h -- C ABI of libmmnn_b200.so (sm_100a kernels for the MMNN_STS training / inference step).
 *
 * Plain pointers and sizes only.  Every pointer is a DEVICE pointer unless it says HOST.  `stream` is a cudaStream_t
 * passed as void*.  Every function that launches work returns 0 on success, a cudaError_t value (> 0) on a CUDA
 * failure or a negative code for an argument the kernels do not support; nothing here allocates or synchronises
 * (except mmnn_profile_collect).  The reference has no FFI of its own (it is a pure PyTorch repository): each entry
 * point below names the reference code it replaces; the Python binding the reference side would use is
 * mmnn_sts_b200/_lib.py (ctypes) and is shown in INTEGRATION.md.
 *
 * Storage formats: forward activations and forward weight images are IEEE fp16 (mmnn_act_is_fp16() == 1),
 * gradient tensors bf16, accumulation / statistics / parameters / losses fp32 (statistics arena fp64).
 */
#ifndef MMNN_B200_H
#define MMNN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------------ trunk (coarse)
 * Replaces DenseNet.backbone: conv0/norm0/relu0/pool0, _DenseBlock x4 of _DenseLayer, _Transition x3, norm5
 * (/root/reference/models/densenet.py:46-148,196-231) and its autograd backward.
 * params / buffers / grads are HOST arrays of device pointers in backbone.named_parameters() / named_buffers() order. */
void* mmnn_encoder_create(int in_channels, const int* block_config /*HOST*/, int nblocks, int init_features,
                          int growth_rate, int bn_size);
void mmnn_encoder_destroy(void* plan);
int mmnn_encoder_num_params(void* plan);
int mmnn_encoder_num_buffers(void* plan);
int mmnn_encoder_num_layers(void* plan);
long long mmnn_encoder_param_numel(void* plan, int index);
int mmnn_encoder_out_channels(void* plan);
long long mmnn_encoder_workspace_bytes(void* plan, int B, int X, int Y, int Z);
int mmnn_encoder_out_dims(void* plan, int B, int X, int Y, int Z, int* out_dhw /*HOST [3]*/);
int mmnn_encoder_debug_offsets(void* plan, int B, int X, int Y, int Z, long long* offs /*HOST*/, long long* dims /*HOST*/);
/* image fp32 NCDHW [B][cin][X][Y][Z];  dropmask fp32 [layers][B][32] keep/(1-p) or NULL;  out fp32 [B*d*h*w][C] NDHWC */
int mmnn_encoder_forward(void* plan, int B, int X, int Y, int Z, const float* image, const void* const* params /*HOST*/,
                         void* const* buffers /*HOST*/, const float* dropmask, void* workspace, float* out, int training,
                         void* stream);
/* Same forward with the image as IEEE fp16 (a data loader that ships 16-bit volumes: half the host->device bytes per step).  The fp32
 * entry point rounds the image to the activation format first thing, so both give the same result for fp16-representable inputs. */
int mmnn_encoder_forward_f16(void* plan, int B, int X, int Y, int Z, const void* image_f16, const void* const* params /*HOST*/,
                             void* const* buffers /*HOST*/, const float* dropmask, void* workspace, float* out, int training,
                             void* stream);
/* grad_out fp32 [B*d*h*w][C];  grads: zero-initialised fp32 tensors shaped like the parameters;  training: the mode of the
 * forward pass that filled `workspace` (batch-statistic or running-statistic BatchNorm is differentiated accordingly) */
int mmnn_encoder_backward(void* plan, int B, int X, int Y, int Z, const void* const* params /*HOST*/,
                          void* const* buffers /*HOST*/, void* const* grads /*HOST*/, const float* dropmask, void* workspace,
                          const float* grad_out, int training, void* stream);

/* Gradient groups for data-parallel overlap (SURVEY.md section 8e: all-reduce overlapped with backward).  Backward
 * finalises the gradients block by block, last block first; group k = dense block (nblocks-1-k) with the transition
 * after it (+ norm5 for k = 0), group nblocks = the stem.  Each group is a contiguous element range [lo, hi) of a
 * buffer that holds all gradients back to back in parameter order (what mmnn_sts_b200.models.densenet passes as
 * `grads`); mmnn_encoder_wait_grad_group makes `stream` wait (cudaStreamWaitEvent) until group k of the most recent
 * mmnn_encoder_backward is final, so its NCCL all-reduce can run while earlier blocks are still in backward. */
int mmnn_encoder_num_grad_groups(void* plan);
int mmnn_encoder_grad_group_range(void* plan, int k, long long* lo /*HOST*/, long long* hi /*HOST*/);
int mmnn_encoder_wait_grad_group(void* plan, int k, void* stream);

/* ------------------------------------------------------------------------------------------------ trunk (fine-grained)
 * The tcgen05 tile engine behind the trunk, exposed for per-kernel parity tests.
 * mmnn_conv_rows  : implicit-GEMM forward / data-gradient of nn.Conv3d 1x1x1, 3x3x3 (pad 1), 7x7x7 (stride 2, pad 3)
 *                   (/root/reference/models/densenet.py:78,82,147,199) with fused BN+ReLU prologue, fused
 *                   per-channel statistics / ReLU-mask epilogue.  amode 0 linear/3x3x3, 1 stem;  trans 0 none,
 *                   1 BN+ReLU;  epi 0 store, 1 store+stats, 2 relu-mask+BN-backward stats;  grad 0 fwd, 1 dgrad.
 * mmnn_conv_wgrad : weight gradient of the same convolutions (kind 0 1x1x1, 1 3x3x3, 2 raw x raw, 3 stem).
 * mmnn_pack_weights: fp32 master weights -> 16-bit k-block images (descs is a HOST array).
 * struct layouts: mmnn_sts_b200/csrc/engine.cuh (RowsParams, WgradParams), pack.cuh (PackDesc); sizes are checked by
 * the mmnn_sizeof_* functions against the ctypes mirrors in mmnn_sts_b200/_lib.py. */
struct RowsParams;
struct BrickParams;
struct WgradParams;
struct PackDesc;
int mmnn_conv_rows(const struct RowsParams* p /*HOST*/, int amode, int trans, int epi, int grad, void* stream);
/* mmnn_conv3_brick: the 3x3x3 forward / data-gradient in "brick mode" (halo brick of a 1x16x8 tile staged once in
 *                   shared memory, taps = descriptor start addresses); used when the spatial dims are >= 8. */
int mmnn_conv3_brick(const struct BrickParams* p /*HOST*/, int grad, void* stream);
int mmnn_sizeof_brick_params(void);
/* mmnn_stem_brick : the stem Conv3d(C_in -> 64, k 7, s 2, p 3) (/root/reference/models/densenet.py:199) in brick mode on
 *                   the padded space-to-depth image (4x4x4 taps over 16 channels, weights resident in shared memory),
 *                   fused per-channel statistics of the stored output for norm0.  StemBrickParams: csrc/stem.cuh. */
struct StemBrickParams;
int mmnn_stem_brick(const struct StemBrickParams* p /*HOST*/, void* stream);
int mmnn_sizeof_stem_brick_params(void);
int mmnn_conv_wgrad(const struct WgradParams* p /*HOST*/, int kind, int split, void* stream);
int mmnn_pack_weights(const struct PackDesc* descs /*HOST*/, int n, void* dev_descs, void* stream);
int mmnn_sizeof_rows_params(void);
int mmnn_sizeof_wgrad_params(void);
int mmnn_sizeof_pack_desc(void);
int mmnn_act_is_fp16(void);

/* ------------------------------------------------------------------------------------------------ heads
 * mmnn_gap_linear_* : DenseNet.features = ReLU -> AdaptiveAvgPool3d(1) -> Flatten -> Linear -> Dropout
 *                     (/root/reference/models/densenet.py:234-247).  y fp32 [B][V][C]; mask [B][F] keep/(1-p) or NULL. */
int mmnn_gap_linear_fwd(const float* y, int B, int V, int C, const float* W, const float* bias, const float* mask, int F,
                        float* pooled, float* out, void* stream);
int mmnn_gap_linear_bwd(const float* y, const float* pooled, int B, int V, int C, const float* W, const float* dout,
                        const float* mask, int F, float* dy, float* dW, float* db, void* stream);
/* mmnn_mlp_heads    : MLP.backbone + MLP.features (/root/reference/models/mlp.py:19-51) and the three output heads of
 *                     MultiModalModel.forward (/root/reference/models/multimodal.py:61-77), forward (backward = 0) or
 *                     backward (1).  MlpArgs: mmnn_sts_b200/csrc/heads.cu. */
struct MlpArgs;
int mmnn_mlp_heads(const struct MlpArgs* args /*HOST*/, int backward, void* stream);
int mmnn_sizeof_mlp_args(void);
/* mmnn_cox_nll      : pycox CoxPHLoss as called from CoxPH (/root/reference/losses/losses.py:6-9), S segments
 *                     (head x class) per launch: loss [S] and dloss/dlog_h [S][N].  CoxArgs: heads.cu. */
struct CoxArgs;
int mmnn_cox_nll(const struct CoxArgs* args /*HOST*/, void* stream);
int mmnn_sizeof_cox_args(void);
/* mmnn_cindex_bootstrap : lifelines concordance_index pair counts as used by getCIndices and the bootstrap loop
 *                     (/root/reference/main.py:106-123,768-887): int64 (correct, tied, pairs) per resample. */
struct CindexArgs;
int mmnn_cindex_bootstrap(const struct CindexArgs* args /*HOST*/, void* stream);
int mmnn_sizeof_cindex_args(void);

/* mmnn_gradcam_maps : the attention maps of MultiModalGradCAM (/root/reference/utils/utils.py:253-344) for a whole
 *                     eval-mode batch in ONE launch, replacing the per-patient, per-class trunk backward: the pooled
 *                     gradient of the last dense layer's conv2 output is computed in closed form from the trunk output y
 *                     (norm5 -> ReLU -> average pool -> feature_layer -> output_head), then the reference's map arithmetic
 *                     (cumulative class re-weighting, cam - min, / max, trilinear align_corners=False up-sampling).
 *                     maps fp32 [B][C][X][Y][Z].  -3 when the C x trunk-voxel cams do not fit shared memory.
 *                     GradcamArgs: heads.cu. */
struct GradcamArgs;
int mmnn_gradcam_maps(const struct GradcamArgs* args /*HOST*/, void* stream);
int mmnn_sizeof_gradcam_args(void);
/* CTAs mmnn_gradcam_maps launches for `args` (each reads its sample's trunk-voxel x 32 activations and signs of y once),
 * for bandwidth accounting; negative: the code mmnn_gradcam_maps would return.  Launches nothing. */
long long mmnn_gradcam_ctas(const struct GradcamArgs* args /*HOST*/);

/* mmnn_bce_logits   : nn.BCEWithLogitsLoss(pos_weight) of the classification path (/root/reference/main.py:148-153):
 *                     elementwise loss and dloss/dlogit for all stacked heads in one launch (targets [N][C] reused by
 *                     every head), plus the per-class tp / fp / fn counters of main.py:226-229 (sigmoid > threshold). */
int mmnn_bce_logits(const float* x, const float* y, const float* pos_weight, long long n, int C, long long y_elems, float* loss,
                    float* grad, float threshold, long long count_elems, int* counts, void* stream);

/* ------------------------------------------------------------------------------------------------ optimiser
 * mmnn_sgd_step     : torch.optim.SGD(momentum, nesterov, weight_decay, dampening 0) as the reference builds it
 *                     (/root/reference/main.py:410-414) and steps it (:479-481), for ALL parameter tensors in one
 *                     launch (one per mmnn_sgd_max_tensors() tensors).  p / g / m: HOST arrays of device pointers to
 *                     the fp32 parameter, gradient and momentum buffer of each tensor, n: HOST array of element counts;
 *                     the table travels as the kernel's parameter, one thread block per mmnn_sgd_chunk_elems() elements.
 *                     Momentum buffers start at zero (== torch's first-step clone). */
int mmnn_sgd_step(void* const* p /*HOST*/, const void* const* g /*HOST*/, void* const* m /*HOST*/,
                  const long long* n /*HOST*/, int ntensors, float lr, float momentum, float weight_decay, int nesterov,
                  void* stream);
/* Same update with {lr, momentum, weight_decay} read from DEVICE memory (float[3]) when the kernel runs: a step captured in a
 * CUDA graph then follows OneCycleLR (which cycles lr and momentum after every optimiser step, /root/reference/main.py:414,480)
 * -- the host rewrites the three floats in place between replays. */
int mmnn_sgd_step_dev(void* const* p /*HOST*/, const void* const* g /*HOST*/, void* const* m /*HOST*/,
                      const long long* n /*HOST*/, int ntensors, const float* hyper /*DEVICE float[3]*/, int nesterov,
                      void* stream);
int mmnn_sgd_chunk_elems(void);
int mmnn_sgd_max_tensors(void);

/* ------------------------------------------------------------------------------------------------ input pipeline
 * mmnn_preprocess_volumes : the deterministic image transforms of the reference's val_transforms / train_transforms
 *                     (/root/reference/main.py:64-92): Normalize(mean, std) (/root/reference/utils/utils.py:346-355)
 *                     -> monai ScaleIntensity() -> monai Resize(spatial_size) ("area" = adaptive average pooling),
 *                     per patient over the whole multi-channel volume.  src fp32 [B][C][X][Y][Z], dst fp32
 *                     [B][C][ox][oy][oz], scratch 2*B uint32. */
int mmnn_preprocess_volumes(const float* src, float* dst, void* scratch, int B, int C, int X, int Y, int Z, int ox, int oy,
                            int oz, float mean, float std, void* stream);

/* mmnn_augment_resample / mmnn_augment_intensity : the RANDOM part of train_transforms (/root/reference/main.py:64-85; MONAI 1.2
 *                     RandRotate / RandAxisFlip / RandZoom composed into ONE affine map and fused with Resize; RandShiftIntensity,
 *                     RandAdjustContrast, RandGaussianSmooth, RandGaussianSharpen, RandHistogramShift, RandGaussianNoise) with
 *                     EXPLICIT per-sample parameters drawn by the caller (mmnn_sts_b200/data/transforms.py TrainTransformsGPU).
 *                     Parity unpinned: the reference as shipped never executes these transforms (DESIGN.md section 9).
 *                     sp: device array of B {float a[9]; float t[3]} (source = A (grid - centre) + centre + t, voxel units);
 *                     prm: device array of B AugIntensity (csrc/augment.cu); smooth_sigma [B][3]; sharpen = sigma1 [B][3],
 *                     sigma2 [B][3], alpha [B]; tmp = 3 volumes of v's size; scratch 2*B uint32. */
int mmnn_preprocess_minmax(const float* src, void* scratch, int B, long long per_image, void* stream);
int mmnn_augment_resample(const float* src, float* dst, void* scratch, const void* sp, int B, int C, int X, int Y, int Z, int ox, int oy,
                          int oz, float mean, float std, void* stream);
int mmnn_augment_intensity(float* v, float* tmp, void* scratch, const void* prm, const float* smooth_sigma, const float* sharpen, int B,
                           int C, int ox, int oy, int oz, int any_smooth, int any_sharpen, void* stream);
int mmnn_sizeof_aug_spatial(void);
int mmnn_sizeof_aug_intensity(void);

/* ------------------------------------------------------------------------------------------------ 3-D ResNet encoder
 * The image-only classification encoder of BASELINE configs[3] (/root/reference/models/resnet.py, SURVEY.md 8f-3) as
 * direct convolutions on channels-last (NDHWC) bf16 tensors; parameters / statistics fp32 / fp64.  RnConvGeom:
 * mmnn_sts_b200/csrc/resnet.cu (18 ints: N Di Hi Wi Cin Do Ho Wo Cout kd kh kw sd sh sw pd ph pw).
 * mmnn_rn_conv        : nn.Conv3d forward (dgrad 0: src = input [fp32 when src_is_f32, C_in = 1: the stem, :10], dst = output,
 *                       stats = fp64 [2][Cout] sum / sum of squares of the stored output, zero-initialised, or NULL) or its
 *                       data gradient (dgrad 1: src = output gradient, dst = input gradient, `add` = optional tensor summed in:
 *                       the identity-residual gradient of BasicBlock.forward :83-95, may alias dst).  w fp32 [Cout][Cin][taps].
 * mmnn_rn_conv_wgrad  : dw [Cout][Cin][taps] += x (*) dy (fp32 atomics, zero-initialise for a fresh gradient).  The fp16 tensor-core
 *                       variant first reduces max|dy| into ONE device-global scratch word (no allocation, no host sync): calls
 *                       on different streams of one device must not overlap (MMNN_RN_WGRAD16=0 selects the variant without it).
 * mmnn_rn_bn_coeffs   : nn.BatchNorm3d coefficient table coef fp32 [4][C] = scale, shift, mean, rstd from the batch statistics
 *                       (training: also the running-statistics update, momentum, unbiased variance) or the running ones.
 *                       C outside 1..64: -2, and nothing is written.
 * mmnn_rn_bn_act      : y = [relu](raw * scale + shift [+ res (res_mode 1) | + res * scale2 + shift2 (res_mode 2)]), then
 *                       nn.Dropout(drop_p) (:156-163) from a counter hash of (seed, element) or an injected uint8 keep-mask.
 * mmnn_rn_act_bwd_reduce / mmnn_rn_bn_bwd_apply : backward of that pass: dz = dy * [y > 0] * post_scale; sums fp64 [3][C] =
 *                       sum dz, sum dz * xhat(raw), sum dz * xhat(raw2); draw (draw2) = BatchNorm backward; dz optionally
 *                       stored (identity residual); dgamma / dbeta written (not accumulated).
 * mmnn_rn_head_fwd/bwd: AdaptiveAvgPool3d(1) -> flatten -> Linear(C -> K) -> sigmoid (:165-170); dW / db accumulate. */
struct RnConvGeom;
int mmnn_sizeof_rn_conv_geom(void);
int mmnn_rn_conv(const struct RnConvGeom* g /*HOST*/, int dgrad, int src_is_f32, const void* src, const float* w, void* dst,
                 const void* add, double* stats, void* stream);
/* BasicBlock.conv1 (64 -> 8, 3x3x3 s1 p1) and the block's 1x1x1 stride-1 down-sample convolution (resnet.py:172-179) on the same
 * input: forward of both in one launch (the 1.08 GB stem activation is read once), and dx = dgrad(conv1) + dgrad(down-sample)
 * in one launch.  Return -9 when the geometry is not that pair: the caller then issues the separate mmnn_rn_conv calls. */
int mmnn_rn_conv_fwd_ds(const struct RnConvGeom* g /*HOST*/, const void* x, const float* w, const float* w_ds, void* y, void* y_ds,
                        double* stats, double* stats_ds, void* stream);
int mmnn_rn_conv_dgrad_ds(const struct RnConvGeom* g /*HOST*/, const void* dy, const float* w, const void* dy_ds, const float* w_ds,
                          void* dx, void* stream);
int mmnn_rn_conv_wgrad(const struct RnConvGeom* g /*HOST*/, int x_is_f32, const void* x, const void* dy, float* dw, void* stream);
int mmnn_rn_bn_coeffs(const double* stats, double count, const float* gamma, const float* beta, float* rmean, float* rvar,
                      long long* nbt, float eps, float momentum, int training, int C, float* coef, void* stream);
int mmnn_rn_bn_act(const void* raw, const float* coef, int res_mode, const void* res, const float* coef2, void* y,
                   long long elems, int C, int relu, float drop_p, unsigned long long seed, const unsigned char* mask,
                   void* stream);
int mmnn_rn_act_bwd_reduce(const void* dy, const void* y, float post_scale, const void* raw, const float* coef,
                           const void* raw2, const float* coef2, double* sums, long long elems, int C, void* stream);
int mmnn_rn_bn_bwd_apply(const void* dy, const void* y, float post_scale, const void* raw, const float* coef, const void* raw2,
                         const float* coef2, const double* sums, double inv_count, int eval_mode, void* draw, void* draw2,
                         void* dz, float* dgamma, float* dbeta, float* dgamma2, float* dbeta2, long long elems, int C,
                         void* stream);
int mmnn_rn_head_fwd(const void* y, int B, int V, int C, const float* W, const float* bias, int K, float* pooled, float* out,
                     void* stream);
int mmnn_rn_head_bwd(const float* dout, const float* out, const float* pooled, const float* W, int B, int V, int C, int K,
                     void* dy, float* dW, float* db, void* stream);

/* ------------------------------------------------------------------------------------------------ instrumentation */
void mmnn_profile_enable(int on);
long long mmnn_launch_count(void);
int mmnn_profile_collect(float* ms /*HOST*/, int* counts /*HOST*/);
/* mmnn_profile_enable(2): records keep the real stream structure (side stream, early start); this returns each launch's class and
 * its start / end in ms relative to the first record (n = records returned, cleared afterwards) */
int mmnn_profile_timeline(int* cls /*HOST*/, float* t0 /*HOST*/, float* t1 /*HOST*/, int cap);

#ifdef __cplusplus
}
#endif
#endif /* MMNN_B200_H */
