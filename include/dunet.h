/* dunet.h -- C ABI of libdunet_b200.so: the B200-native Diff-UNet DDIM sliding-window inference path.
 *
 * The reference (aarchiiive/diff-unet-amos) has no FFI of its own: its seams are Python objects (SURVEY.md 8b).
 * Each entry point below names the reference interface it replaces (file:line under /root/reference) -- this is what
 * a ctypes/cffi binding on the reference side binds (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success and a negative DUNET_E_* code on failure; dunet_last_error() returns a
 *     thread-local human-readable message for the last failure on the calling thread.  Nothing throws across the ABI.
 *   - the CALLER owns every buffer (inputs, outputs, workspace).  A plan owns only packed weights, the time-embedding
 *     table, the DDIM coefficient tables, two internal streams + events (DUNET_FLAG_DUAL_STREAM) and a few hundred bytes
 *     of pinned staging for per-sample timesteps -- all created by dunet_plan_commit().  No hidden allocation after
 *     dunet_plan_commit() (exception: with dunet_profile_enable the profiler grows its event pool), no hidden
 *     synchronisation: all work is enqueued on the caller's stream (a cudaStream_t passed as void*).
 *   - device pointers must be 16-byte aligned; the workspace pointer 256-byte aligned (checked).
 *   - boundary tensors are fp32, NCDHW, contiguous -- the reference's layout.  bf16 channels-last staging is internal.
 *   - a plan is not thread-safe (one plan per GPU / stream); distinct plans are independent (profiler state is per
 *     plan; per-device kernel attributes are set once per device under a mutex; the only process-global state is the
 *     dunet_debug_set_conv_timeline hook and the launch counter).
 *   - there is NO CPU fallback: every function that computes requires a CUDA device of compute capability 10.x.
 */
#ifndef DUNET_H_
#define DUNET_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DUNET_VERSION 230 /* 0.2.3; _lib.DUNET_VERSION must match */

/* dunet_cfg.in_channels range.  The encoder's first conv packs the image as [hi | lo | hi] into ONE 32-channel block
 * (3 * in_channels <= 32), and the denoiser input [x_0 .. x_{C-1}, image ..] is packed into 32 channels
 * (num_classes + in_channels <= 32).  Outside these bounds dunet_plan_create returns DUNET_E_UNSUPPORTED. */
#define DUNET_MAX_IN_CHANNELS 10

enum {
  DUNET_OK = 0,
  DUNET_E_INVALID = -1,   /* bad argument / shape / alignment */
  DUNET_E_CUDA = -2,      /* CUDA runtime or driver error (message carries the CUDA error string) */
  DUNET_E_STATE = -3,     /* call order violated (weights missing, plan not committed, ...) */
  DUNET_E_UNSUPPORTED = -4 /* configuration outside what the kernels implement */
};

/* dunet_cfg.flags */
#define DUNET_FLAG_REF_CONV 1u /* debug: run 3x3x3 convs on the CUDA-core reference kernel instead of tcgen05 (tests) */
#define DUNET_FLAG_KEEP_FP32_WEIGHTS 2u /* debug: keep fp32 copies of conv weights (needed by DUNET_FLAG_REF_CONV) */

#define DUNET_FLAG_GENERIC_CONV 4u /* debug: every 3x3x3 / transposed conv on the generic voxel-as-M tcgen05 kernel (no Cout = 64
                                     z-stacked kernel, no flattened-plane kernel for the deep levels) */

#define DUNET_FLAG_DUAL_STREAM 8u /* batches of >= 4 windows run as two half batches on two internal streams (forked from /
                                    joined into the caller's stream with events, no host synchronisation): the HBM-bound
                                    kernels of one half overlap the tensor-bound convolutions of the other.  Measured +3 %
                                    at batch 4 and 8; results are bit-identical (batching is transparent).  Not used while
                                    dunet_profile_enable(1) is active (per-kernel timings would overlap) */

#define DUNET_FLAG_FP32X3 16u /* fp32-class precision mode ("fp32x3", SURVEY 8b/8d): every activation and weight is a
                                 hi + lo pair of bf16 tensors and each product is formed as hi*hi + lo*hi + hi*lo on the
                                 same tcgen05 kernels (3x the MMA work, 2x the activation traffic, fp32 accumulation and
                                 fp32 elementwise math as in bf16 mode).  Meets north_star's 1e-4 / 99.9 % argmax gates */

#define DUNET_FLAG_NO_FUSED_NORM 32u /* debug / A-B timing: materialise the normalised intermediate of every TwoConv with
                                       norm_act_kernel.  By default the second conv of a TwoConv (Cout = 64 kernel, bf16
                                       mode) normalises the first conv's raw output ON LOAD: eight extra warps rewrite each
                                       TMA-loaded halo plane in shared memory (InstanceNorm + LeakyReLU + time bias) before
                                       the MMAs read it, so that tensor never exists in HBM.  Bit-identical results (tested);
                                       64->64 @96^3 x4: 558 us instead of 532 + 157 us */

#define DUNET_FLAG_FP16 128u /* 16-bit storage format of activations and packed weights is IEEE fp16 (11 mantissa bits) instead of
                               bf16 (8): the reference's own reduced precision (torch.autocast fp16, test.py:104,119 with
                               cfg/btcv/test.yaml:16, cfg/msd/test.yaml:16).  Same kernels, same speed (tcgen05 kind::f16 takes
                               F16 operands at the BF16 rate), fp32 accumulation / statistics / DDIM state as in bf16 mode.
                               Range: conv outputs are stored before normalisation, |x| must stay below 65504 (the reference's
                               AMP path has the same limit).  Mutually exclusive with DUNET_FLAG_FP32X3 */

#define DUNET_FLAG_PLAIN_ENCODER 256u /* A-B measurements: with DUNET_FLAG_FP16 the image ENCODER runs in split precision (bf16
                               hi + lo pairs, 3 MMAs per product, like DUNET_FLAG_FP32X3) because its feature maps are added
                               into the denoiser at every level of every DDIM step: its rounding error is the one source that
                               repeats identically in all N steps (2/3 of the fp16 error variance of a window).  The encoder
                               is 2.6 % of the FLOPs.  This flag runs the encoder in plain fp16 as well */

#define DUNET_FLAG_TC64_CB64 64u /* debug / A-B timing: the Cout = 64 kernel walks 64-channel blocks with a 7-slot plane ring
                                   instead of 32-channel blocks with a 13-slot ring */

typedef struct dunet_plan dunet_plan;

/* Mirrors DiffUNet.__init__(spatial_dims=3, in_channels, out_channels, image_size, spatial_size, features, ...)
 * (models/diff_unet.py:10-21) plus the sampler settings hard-coded in Diffusion.__init__
 * (models/diffusion/diffusion.py:38-45: 10 respaced DDIM steps). */
typedef struct dunet_cfg {
  int32_t num_classes;  /* out_channels C; the denoiser input has in_channels + C channels (denoiser.py:298) */
  int32_t in_channels;  /* image channels (modalities), 1 .. DUNET_MAX_IN_CHANNELS with num_classes + in_channels <= 32 */
  int32_t patch[3];     /* window (D, H, W); each a multiple of 16 and >= 32 (SURVEY 8c) */
  int32_t features[6];  /* models/diff_unet.py:17, default {64,64,128,256,512,64} */
  int32_t batch_max;    /* windows processed together (the reference loops at batch 1, diffusion.py:88-89) */
  int32_t num_steps;    /* DDIM steps N of space_timesteps(1000, [N]) */
  uint32_t flags;
} dunet_cfg;

int dunet_version(void);
const char* dunet_last_error(void);

/* replaces: DiffUNet(...) construction, models/diff_unet.py:9-35 */
int dunet_plan_create(dunet_plan** out, const dunet_cfg* cfg);
void dunet_plan_destroy(dunet_plan* plan);

/* replaces: model.load_state_dict(torch.load(path)['model']), test.py:85-91.  `key` is the reference checkpoint key
 * (SURVEY Appendix F, e.g. "model.upcat_4.upsample.deconv.weight"); `dev_ptr` an fp32 device tensor in the reference's
 * own layout ([Cout,Cin,3,3,3] convs, [Cin,Cout,2,2,2] transposed convs).  The plan re-packs into its kernel layout. */
int dunet_plan_set_weight(dunet_plan* plan, const char* key, const float* dev_ptr, const int64_t* shape, int32_t ndim,
                          void* stream);

/* replaces: SpacedDiffusion tables + _WrappedModel timestep map (guided_diffusion/respace.py:72-86,123-129;
 * gaussian_diffusion.py:131-147).  Host arrays of length n_steps; the float tables are the float64 tables cast to fp32
 * exactly as _extract_into_tensor does (gaussian_diffusion.py:914). */
int dunet_plan_set_schedule(dunet_plan* plan, int32_t n_steps, const int32_t* timestep_map,
                            const float* sqrt_recip_alphas_cumprod, const float* sqrt_recipm1_alphas_cumprod,
                            const float* alphas_cumprod_prev);

/* Validates that all weights + schedule are present and builds the per-(step, TwoConv) time-embedding bias table
 * (TimeStepEmbedder + temb_proj, models/diffusion/utils.py:31-54, denoiser.py:51-52,65). */
int dunet_plan_commit(dunet_plan* plan, void* stream);

int dunet_workspace_bytes(const dunet_plan* plan, int32_t batch, size_t* out_bytes);

/* replaces: BasicUNetEncoder.forward(image), models/basic_unet/pretrained/basic_unet.py:496-512.
 * image: [batch, in_channels, D, H, W] fp32.  The five feature maps stay in the workspace (bf16) for the denoiser. */
int dunet_encode(dunet_plan* plan, const float* image, int32_t batch, void* workspace, void* stream);
/* copies feature map `level` (0..4) out as fp32 NCDHW [batch, features[level], D>>level, ...] / back in */
int dunet_get_embedding(dunet_plan* plan, int32_t level, float* out, int32_t batch, void* workspace, void* stream);
int dunet_set_embedding(dunet_plan* plan, int32_t level, const float* in, int32_t batch, void* workspace, void* stream);

/* replaces: BasicUNetRDenoiser.forward(x, t, image=, embeddings=), models/basic_unet/denoiser.py:284-312, as called
 * from GaussianDiffusion.p_mean_variance (gaussian_diffusion.py:259) and from Diffusion.denoise (training forward,
 * models/diffusion/diffusion.py:71-84, train.py:258-268).  `t_original`: HOST array of `batch` ORIGINAL timesteps (after
 * the respace remap), one per sample.  When all are equal and a member of the plan's schedule (the inference call) the
 * precomputed time-embedding row is used; otherwise a per-sample bias table is built for this call (the timesteps are
 * staged through plan-owned pinned memory, nothing is allocated).  Embeddings are those left in the workspace by
 * dunet_encode / dunet_set_embedding.  x_t: [batch, C, D, H, W], image: [batch, in_channels, D, H, W], logits_out:
 * [batch, C, D, H, W], all fp32. */
int dunet_denoise_step(dunet_plan* plan, const float* x_t, const float* image, const int32_t* t_original,
                       float* logits_out, int32_t batch, void* workspace, void* stream);

/* replaces: Diffusion.ddim_sample(image) for a batch of windows (models/diffusion/diffusion.py:86-102), i.e.
 * embed_model + SpacedDiffusion.ddim_sample_loop (gaussian_diffusion.py:626-716) + the sum of the N clamped x0
 * predictions.  image: [batch, in_channels, D, H, W] fp32; noise: [batch, C, D, H, W] fp32 initial x_T (gaussian_diffusion.py:690-693); acc_out receives
 * sum_k clamp(model_output_k, -1, 1); per_step_logits (nullable): [n_steps, batch, C, D, H, W] raw model outputs in
 * loop order (t high -> low); final_x (nullable): the last sample.  run_encoder == 0 skips the encoder and uses the
 * embeddings already in the workspace (the reference's ddim_sample_loop(model, shape, model_kwargs={image, embeddings})
 * seam, gaussian_diffusion.py:626-665).  Ensemble averaging over R independent noise draws (BASELINE config 4): call R times
 * with out_scale = 1/R, out_accumulate = 0 for the first draw and 1 afterwards (acc_out = [acc_out +] out_scale * sum_k x0_k);
 * the reference itself corresponds to out_scale = 1, out_accumulate = 0. */
int dunet_ddim_sample(dunet_plan* plan, const float* image, const float* noise, float* acc_out, float* per_step_logits,
                      float* final_x, int32_t batch, int32_t run_encoder, float out_scale, int32_t out_accumulate,
                      void* workspace, void* stream);

/* replaces: the body of monai.inferers.sliding_window_inference as called at engine.py:173-177 (constant blend):
 * window crop, `out[slices] += pred`, `out /= count`, and Engine.infer's sigmoid+threshold (engine.py:179-180). */
int dunet_crop_window(const float* volume, const int32_t vol_dims[3], float* patch, const int32_t patch_dims[3],
                      const int32_t start[3], void* stream);
int dunet_stitch_add(float* out_volume, const int32_t vol_dims[3], int32_t channels, const float* patch,
                     const int32_t patch_dims[3], const int32_t start[3], void* stream);
/* replaces: `output_image = torch.zeros(...)` at the start of sliding_window_inference: clears the caller's accumulator
 * (cudaMemsetAsync on `stream`; no kernel launch). */
int dunet_zero(void* ptr, size_t bytes, void* stream);
/* all windows of a batch in one launch: patches[b] = volume[start_b : start_b + patch_dims]; starts: HOST [batch][3].
 * dunet_crop_window(s) take ONE channel ([D, H, W] volume); crop a multi-channel volume channel by channel. */
int dunet_crop_windows(const float* volume, const int32_t vol_dims[3], float* patches, const int32_t patch_dims[3],
                       const int32_t* starts, int32_t batch, void* stream);

/* replaces: ONE iteration of the window loop of sliding_window_inference with predictor = Diffusion.forward(pred_type=
 * "ddim_sample") (engine.py:173-177 + models/diffusion/diffusion.py:86-102): crop `batch` windows out of `volume`
 * ([in_channels, D, H, W] fp32, already padded to >= the plan's patch), run encoder + N DDIM steps on them, and add the results into
 * `out_volume` ([C, D, H, W] fp32) window by window in the given order -- `out[slices] += pred`, bit-identical to
 * dunet_crop_window + dunet_ddim_sample + dunet_stitch_add, without the planar [batch, C, patch] intermediates.
 *   starts     HOST [batch][3] window corners (MONAI order)
 *   noise      nullable device [ensemble][batch][C][patch] fp32: the initial x_T (parity runs).  NULL: the library draws
 *              N(0,1) itself with a counter-based generator (Philox4x32-10, Box-Muller) keyed by (seed, noise_ids[b],
 *              draw): a window's noise does not depend on batching, rank or launch order
 *   noise_ids  HOST [batch] stream id per window (e.g. its global index in the volume's window list); needed if noise == NULL
 *   ensemble   R >= 1 independent draws averaged (BASELINE config 4; R = 1 is the reference)
 *   weights / count_volume   both NULL: constant blend.  Otherwise MONAI mode="gaussian": out += w * pred, count += w.
 * With DUNET_FLAG_DUAL_STREAM the two half batches run on the plan's internal streams, forked from and joined back into
 * `stream`; the stitching then runs on `stream` in window order.  Everything is ordered on `stream` when the call returns. */
int dunet_infer_windows(dunet_plan* plan, const float* volume, const int32_t vol_dims[3], const int32_t* starts,
                        int32_t batch, const float* noise, uint64_t seed, const int64_t* noise_ids, int32_t ensemble,
                        float* out_volume, float* count_volume, const float* weights, void* workspace, void* stream);
/* counts_d/h/w: device int32 arrays, number of windows covering each coordinate along that axis (the window grid is a
 * Cartesian product so count(z,y,x) = counts_d[z]*counts_h[y]*counts_w[x]).  binary/argmax_labels nullable. */
int dunet_finalize(float* out_volume, const int32_t vol_dims[3], int32_t channels, const int32_t* counts_d,
                   const int32_t* counts_h, const int32_t* counts_w, uint8_t* binary, uint8_t* argmax_labels,
                   void* stream);

/* Multi-GPU: the exchange of the per-rank partial volumes FUSED with dunet_finalize, over NVLink peer memory.  The calling
 * rank owns channels [channel_lo, channel_hi).  partial_ptrs (HOST array of n_src device pointers, each the [C, D, H, W] fp32
 * partial sum volume of one contributing rank -- its own memory or a CUDA-IPC peer mapping) are read directly by the kernel;
 * source k is only read for dim-0 rows [slab_lo[k], slab_hi[k]) (the slab its windows touched, HOST arrays).  The kernel
 * adds the contributions in array order, divides by the coverage counts, binarises and stores the uint8 labels (and, if
 * `blended` is non-NULL, the normalised fp32 logits) into `binary` / `blended`, which may live on another GPU as well.
 * Replaces ncclReduceScatter + dunet_finalize + gather; cross-rank ordering (all partial sums complete before, all reads
 * complete after) is the caller's job (dist.py uses two tiny NCCL all-reduces per window-queue group as stream barriers). */
int dunet_finalize_peers(const float* const* partial_ptrs, const int32_t* slab_lo, const int32_t* slab_hi, int32_t n_src,
                         const int32_t vol_dims[3], int32_t channel_lo, int32_t channel_hi, const int32_t* counts_d,
                         const int32_t* counts_h, const int32_t* counts_w, uint8_t* binary, float* blended, void* stream);

/* CUDA-IPC plumbing for dunet_finalize_peers (one process per GPU): dunet_ipc_alloc = cudaMalloc + cudaIpcGetMemHandle
 * (the 64-byte handle travels to the other ranks through torch.distributed), dunet_ipc_open maps another rank's buffer into
 * this process with NVLink peer access enabled, dunet_ipc_close / dunet_ipc_free undo them. */
int dunet_ipc_alloc(void** ptr, size_t bytes, uint8_t handle_out[64]);
int dunet_ipc_open(const uint8_t handle[64], void** ptr);
int dunet_ipc_close(void* ptr);
int dunet_ipc_free(void* ptr);

/* MONAI blend mode "gaussian" (SURVEY 8f-4; the reference's own call uses the default constant blend): out[slices] += w * pred
 * and count[slices] += w with `weights` the [pd0, pd1, pd2] fp32 importance map of a window; dunet_finalize_weighted divides
 * by the accumulated fp32 count volume [D, H, W] and binarises like dunet_finalize. */
int dunet_stitch_add_weighted(float* out_volume, float* count_volume, const int32_t vol_dims[3], int32_t channels,
                              const float* patch, const float* weights, const int32_t patch_dims[3], const int32_t start[3],
                              void* stream);
int dunet_finalize_weighted(float* out_volume, const float* count_volume, const int32_t vol_dims[3], int32_t channels,
                            uint8_t* binary, uint8_t* argmax_labels, void* stream);

/* replaces: monai.transforms.ScaleIntensityRanged(a_min=-175, a_max=250, b_min=0, b_max=1, clip=True), the intensity step
 * of the reference's val/test transforms (utils.py:167-170, 185-187), as a GPU pre-pass feeding the window driver
 * (SURVEY 8f-3).  y = (x - a_min) / (a_max - a_min) * (b_max - b_min) + b_min, optionally clipped; in == out allowed. */
int dunet_scale_intensity(const float* in, float* out, int64_t n, float a_min, float a_max, float b_min, float b_max,
                          int32_t clip, void* stream);

/* replaces: monai.transforms.CropForegroundd(keys=["image", "label"], source_key="image") of the reference's val transforms
 * (utils.py:171).  dunet_foreground_bbox writes {min z, min y, min x, max z + 1, max y + 1, max x + 1} of the voxels with
 * image > 0 (any channel; MONAI generate_spatial_bounding_box with select_fn = is_positive, margin 0) to the DEVICE array
 * bbox_dev[6]; an all-background image gives {D, H, W, 0, 0, 0}.  dunet_crop_box is the SpatialCrop applied to image and
 * label: out[c] = in[c][start : start + out_dims].  Exact (integer / copy). */
int dunet_foreground_bbox(const float* image, int32_t channels, const int32_t dims[3], int32_t* bbox_dev, void* stream);
int dunet_crop_box(const float* in, int32_t channels, const int32_t dims[3], float* out, const int32_t out_dims[3],
                   const int32_t start[3], void* stream);
/* replaces: monai.transforms.Spacingd(pixdim=(1.5, 1.5, 2.0), mode=("bilinear", "nearest")) (utils.py:173-177) for
 * axis-aligned affines: out[c][i, j, k] = sample(in[c], (i * ratio[0], j * ratio[1], k * ratio[2])), ratio = new / old
 * spacing per axis, coordinates clamped to the border; mode 0 trilinear (image), 1 nearest (label).  The caller sizes
 * `out` as round((dim - 1) / ratio) + 1 per axis (MONAI compute_shape_offset).  Interpolation in fp32 in a fixed order. */
int dunet_resample_spacing(const float* in, int32_t channels, const int32_t dims[3], float* out, const int32_t out_dims[3],
                           const double ratio[3], int32_t mode, void* stream);

/* replaces: MONAI Invertd(keys="pred", transform=val_transforms, orig_keys="image") of the val transforms' Spacingd +
 * CropForegroundd (utils.py:171-177), followed by AsDiscreted / the binarisation of engine.py:179-180: labels on the grid of
 * the array the val transforms received, in one pass, without fp32 intermediates on that grid.
 *   blended   the finalised fp32 [channels][vol_dims] volume (dunet_finalize / dunet_finalize_weighted leave it divided by
 *             the coverage); the resampled volume [res_dims] lies at `offset` inside it (the window driver pads a volume
 *             smaller than the roi: offset = (vol - res) / 2 per axis, floor).
 *   out_dims  the original grid (D0, H0, W0); the foreground box [box_start, box_start + box_dims) lies inside it and has
 *             the shape the forward crop produced (the forward resample went box_dims -> res_dims).
 * For every output voxel p: outside the box binary = 0 and argmax = 0 (MONAI's inverse BorderPad inserts zero logits).
 * Inside, with j = p - box_start, the sample coordinate on axis d is clamp(j_d * ratio[d], 0, res_dims[d] - 1), formed in
 * fp64, ratio = spacing_in / pixdim (the inverse of dunet_resample_spacing's pixdim / spacing_in); mode 0 nearest (index
 * rint(coordinate), Invertd's default nearest_interp=True), 1 trilinear (fp32 lerps in dunet_resample_spacing's order).
 * Then binary[c][p] = sigmoid(logit_c) > 0.5 and argmax[p] = first maximum over classes, as dunet_finalize forms them: the
 * result is bit-identical to dunet_resample_spacing to box_dims, zero padding to out_dims and dunet_finalize with unit counts.
 * binary [channels][out_dims] or NULL, argmax [out_dims] or NULL (not both; channels <= 256 with argmax); ratios finite > 0. */
int dunet_invert_labels(const float* blended, int32_t channels, const int32_t vol_dims[3], const int32_t offset[3],
                        const int32_t res_dims[3], const double ratio[3], const int32_t box_start[3],
                        const int32_t box_dims[3], const int32_t out_dims[3], int32_t mode,
                        uint8_t* binary, uint8_t* argmax, void* stream);

/* Uncertainty-weighted fusion of the DDIM steps of `runs` independent sampling runs (the test-time fusion of upstream
 * Diff-UNet; this reference returns the plain sum instead, models/diffusion/diffusion.py:94-98; SURVEY 8f-4).
 * per_step: [runs][n_steps][n] fp32 raw model outputs in loop order (per_step_logits of dunet_ddim_sample);
 * out[n] = sum_k exp(sigmoid((k + 1) / n_steps) * (1 - u_k)) * sum_r clamp(per_step[r][k], -1, 1) with
 * u_k = -p log p, p = max(sigmoid(mean_r per_step[r][k]), 0.001). */
int dunet_uncertainty_fuse(const float* per_step, int32_t runs, int32_t n_steps, int64_t n, float* out, void* stream);

/* replaces: GaussianDiffusion.q_sample (gaussian_diffusion.py:187-205) as Diffusion.q_sample calls it in the training forward
 * (models/diffusion/diffusion.py:65-69, train.py:258-268): out[n] = sqrt_ac[t[n]] * x_start[n] + sqrt_1mac[t[n]] * noise[n].
 * x_start / out: [batch][per_sample] fp32; t_dev: DEVICE int64 [batch]; sqrt_ac / sqrt_1mac: DEVICE fp32 tables of the
 * training schedule (float64 tables cast to fp32 like _extract_into_tensor, :914).  noise_in NULL: N(0,1) noise is drawn by
 * the library generator (stream ids id0 + n) and returned in noise_out.  Bit-identical to the torch expression. */
int dunet_q_sample(const float* x_start, const float* noise_in, float* noise_out, const int64_t* t_dev, const float* sqrt_ac,
                   const float* sqrt_1mac, float* out, int32_t batch, int64_t per_sample, uint64_t seed, int64_t id0,
                   void* stream);

/* replaces: the per-class reductions of dice_coeff (metric.py:3-49) as Tester.validation_step calls it on the binarised
 * volume (test.py:143-151).  pred: uint8 {0,1} [channels][voxels] (dunet_finalize's `binary`); label: one-hot
 * [channels][voxels], uint8 or fp32 (label_is_float), non-zero = foreground.  counts (device, [channels][3] uint64):
 * { |pred & label|, |pred|, |label| } -- exact integers; the Dice value and the reference's special cases
 * (pred non-empty & label empty -> 1; both empty -> 0) are host arithmetic on these. */
int dunet_dice_counts(const uint8_t* pred, const void* label, int32_t label_is_float, int32_t channels, int64_t voxels,
                      uint64_t* counts, void* stream);

/* replaces: medpy.metric.binary.hd95(result, reference, voxelspacing, connectivity=1) per class, in the reference's
 * medpy-based evaluation (metric module, SURVEY row 12; the call is commented out in test.py:153-158).  pred and label
 * as in dunet_dice_counts, laid out [channels][D][H][W] with dims = (D, H, W); spacing[d] is medpy's voxelspacing of
 * array axis d (finite, > 0).  hd95_out (device fp64 [channels]) gets per class, with A = pred, B = label:
 *   border(M) = M ^ binary_erosion(M, 6-connected, border_value 0)   (voxels on the volume edge are border voxels);
 *   d_AB      = distance_transform_edt(~border(B), sampling=spacing)[border(A)], d_BA likewise;
 *   HD95      = numpy.percentile(d_AB ++ d_BA, 95), default linear method.
 * Each distance is formed from the integer offset to the nearest site as sqrt(((s0 d0)^2 + (s1 d1)^2) + (s2 d2)^2) in fp64,
 * as scipy forms it, and the interpolation is numpy's _lerp without FMA: the result is bit-identical to the scipy / numpy
 * computation whenever the squared terms are exact in fp64 (e.g. spacings that are multiples of 0.25 mm).
 * A class whose prediction or label is empty gets NaN (medpy raises); the other classes are unaffected.
 * Workspace: dunet_hd95_workspace_bytes, 24 bytes per voxel plus 4 KB, independent of the class count (classes run one
 * after another); 256-byte aligned.  Alignment: an fp32 label 4 bytes, hd95_out 8 bytes, pred and a uint8 label none (per-sample
 * slices of a batch can be passed as they are).  Per class 17 kernel launches: state init, bounding box of pred ∪ label with the
 * border counts, three separable passes per direction restricted to that box, eight radix-select passes and the
 * percentile.  No host synchronisation.  dims must be in [1, 32767] (DUNET_E_UNSUPPORTED above). */
int dunet_hd95_workspace_bytes(int32_t channels, const int32_t dims[3], size_t* out_bytes);
int dunet_hd95(const uint8_t* pred, const void* label, int32_t label_is_float, int32_t channels, const int32_t dims[3],
               const double spacing[3], double* hd95_out, void* workspace, size_t workspace_bytes, void* stream);

/* Stand-alone operator (also the unit-test seam of the tensor-core kernel): y = conv3d(cat([src0, src1]), weight),
 * 3x3x3, stride 1, zero padding 1, no bias.  fp32 NCDHW in/out, bf16 operands + fp32 accumulation inside.
 * use_ref_kernel: 0 = production tcgen05 kernels, 1 = CUDA-core debug kernel, 2 = generic tcgen05 kernel only,
 * 3 / 4 = as 0 / 2 in fp32x3 mode (operands split into hi + lo bf16 pairs, see DUNET_FLAG_FP32X3),
 * 5 / 6 = as 0 / 2 with fp16 operands (DUNET_FLAG_FP16).
 * The kernel is chosen as for a plan's layer at these dims, except that this operator never splits K: a layer that a
 * plan runs K-split (ksplit > 1 in dunet_debug_conv_geometry) runs here unsplit -- with Cout <= 64 that can mean the
 * z-stacked kernel where the plan runs the generic one.
 * replaces: nn.Conv3d inside MONAI Convolution (denoiser.py:56-58).  use_ref_kernel != 0 selects the debug CUDA-core
 * kernel.  Allocates its own scratch with cudaMallocAsync on `stream`. */
int dunet_op_conv3x3x3(const float* src0, int32_t c0, const float* src1, int32_t c1, const float* weight, int32_t cout,
                       float* out, int32_t batch, const int32_t dims[3], int32_t use_ref_kernel, void* stream);

/* Stand-alone transposed convolution k=2 s=2 + bias: y = conv_transpose3d(src, weight[cin, cout, 2, 2, 2], bias).
 * replaces: nn.ConvTranspose3d inside MONAI UpSample(mode="deconv") (denoiser.py:161-170, 181).  fp32 NCDHW in/out. */
int dunet_op_deconv2x2x2(const float* src, int32_t cin, const float* weight, const float* bias, int32_t cout, float* out,
                         int32_t batch, const int32_t dims[3], int32_t use_ref_kernel, void* stream);

/* Host-only (no CUDA call, works without a GPU): the kernel and tiling a 3x3x3 conv layer cin -> cout gets on a U-Net level of
 * dims = (D, H, W) voxels per sample under plan flags `flags` -- the plan's own decision, read from the same function that the
 * layer launches and the workspace size read.  The decision is a function of per-sample shapes only (never of
 * the batch), which is what keeps batching bit-transparent.  out[16] = { kernel (0 = Cout-64 z-stacked conv3d_tc64, 1 = generic
 * voxel-as-M conv3d_tc, 2 = flattened-plane conv3d_flat), zt, tiles_x, tiles_y, tiles_z, ksplit, K units per 64-channel block
 * (1 or 3), hx, ty, npos, plane-ring slots, weight-ring slots, dynamic shared memory bytes (kernel 2), work items per sample and
 * K split, cout tiles, 64-channel input blocks }.  Fields 7-12 are 0 unless kernel == 2.  Under DUNET_FLAG_REF_CONV the
 * CUDA-core kernel runs; it reports kernel 1 and the generic kernel's tiling, from which the workspace is sized. */
int dunet_debug_conv_geometry(const int32_t dims[3], int32_t cin, int32_t cout, uint32_t flags, int32_t out[16]);

/* tools only: when non-NULL every conv CTA writes 8 clock64 stamps to dev_buffer[cta * 8 ..] (kernel start, first MMA
 * batch issued, last MMA committed, accumulators complete, epilogue done).  PROCESS-GLOBAL debugging hook (the one
 * piece of library state that is not per plan): it applies to every plan's generic conv launches until reset.
 * DUNET_DBG_LAUNCH=k in the environment restricts the stamps to the k-th generic / flattened-plane conv launch since the hook
 * was set; DUNET_DBG_DECONV=1 lets the persistent transposed-conv kernel write them as well.  Neither changes a result. */
int dunet_debug_set_conv_timeline(int64_t* dev_buffer);

/* Live kernel timing for bench.py's roofline, PER PLAN: when enabled, every launch this plan makes is bracketed by CUDA
 * events on the launching stream (and DUNET_FLAG_DUAL_STREAM is suspended so kernel times do not overlap).
 * dunet_profile_read synchronises those events and returns, since the last enable: summed conv kernel time (ms), number
 * of conv launches, and their ALGORITHMIC flops 2*B*V*Cout*27*Cin (real channels only). */
int dunet_profile_enable(dunet_plan* plan, int32_t on);
int dunet_profile_read(dunet_plan* plan, double* conv_ms, uint64_t* conv_launches, double* conv_flops);
/* per kernel family, arrays of 12 entries: 0 conv3x3x3 (16-bit operands; also fp32x3 plans), 1 normalise (launches moving
 * >= 64 MB), 2 final+DDIM, 3 transposed conv, 4 split-K reduce, 5 other (affine-map kernel), 6 normalise launches below 64 MB
 * (launch-latency bound), 7 glue (window crop, noise + state init, stitch), 8 conv3x3x3 running in split precision inside a
 * 16-bit plan (the encoder in fp16 mode: 3 MMAs per algorithmic product), 9 transposed-conv launches below 64 MB (tag 3 then
 * holds the launches >= 64 MB), 10-11 unused.  For the two conv families
 * bytes_by_tag holds ALGORITHMIC FLOPs instead of bytes.
 * bytes_by_tag (nullable): ALGORITHMIC HBM bytes of the bandwidth-bound families (normalise: 4 B/element (+2 residual,
 * +0.25 pooled); final+DDIM: per voxel 2F + 16C (+2C re-pack); transposed conv: 2(Cin + 8 Cout) per input voxel). */
int dunet_profile_read_all(dunet_plan* plan, double* ms_by_tag, uint64_t* launches_by_tag, double* bytes_by_tag);
/* every profiled launch in issue order: duration (ms) and kernel family tag */
int dunet_profile_dump(dunet_plan* plan, double* ms, int32_t* tags, int32_t capacity, int32_t* count);

/* Device-side pipeline watchdog: non-zero if a bounded mbarrier wait expired inside a kernel (kernel bug). */
int dunet_debug_barrier_timeouts(uint32_t* out_flag);
/* Number of kernels this library has launched on the calling process since load (bench.py's gpu_launches). */
uint64_t dunet_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* DUNET_H_ */
