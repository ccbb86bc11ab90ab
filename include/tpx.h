/* libtpx_b200 — C ABI of the B200-native 3DTopia-XL denoising hot path (DiT step, sampler update, VAE decode).
 *
 * The reference has NO C/FFI interface for this path: its boundary is a set of Python objects resolved by
 * dva/io.py:22-28 (`load_from_config`).  Each entry point below therefore cites the reference *Python*
 * interface it stands behind; the Python mirror of those interfaces (3dtopia-xl_b200/{dit,diffusion,vae}.py)
 * is a thin ctypes caller of this header.  INTEGRATION.md shows the binding a maintainer adds.
 *
 * Conventions: plain pointers and sizes only; every pointer named *dev* / documented "device" is a CUDA
 * device pointer on the current device; `stream` is a cudaStream_t passed as void* (NULL = legacy default
 * stream); all work is enqueued asynchronously on that stream, no host synchronisation, no allocation
 * inside hot calls (workspaces are caller-allocated, sizes from *_workspace_bytes); functions return 0 or a
 * negative TPX_ERR_* code and never throw; tpx_last_error() gives the thread-local message.
 * Handles are not thread-safe; distinct handles are independent.  Device code is sm_100a only: every entry
 * that launches work fails with TPX_ERR_CUDA on any other device — there is no CPU or other-arch fallback.
 */
#ifndef TPX_B200_H
#define TPX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TPX_VERSION 100 /* 0.1.0 */

enum { TPX_OK = 0, TPX_ERR_ARG = -1, TPX_ERR_CUDA = -2, TPX_ERR_SHAPE = -3, TPX_ERR_STATE = -4, TPX_ERR_KEY = -5 };
enum { TPX_DTYPE_F32 = 0, TPX_DTYPE_F16 = 1 };

int tpx_version(void);
const char* tpx_last_error(void);
/* 0 if the current device can run the kernels (compute capability 10.x), else TPX_ERR_CUDA. */
int tpx_device_check(void);
/* Measurement hooks (bench.py): total kernels launched by this library so far; and an optional mode that brackets
 * every launch with a CUDA event pair on its stream.  profile_end synchronises the device and returns, per kernel
 * class, the summed device time (ms) and launch count.  Classes: 0 tcgen05 GEMM, 1 attention, 2 LayerNorm+modulate,
 * 3 GEMV/embedders, 4 CFG/sampler, 5 implicit-GEMM conv, 6 GroupNorm, 7 other VAE. */
#define TPX_PROF_NCLASS 8
int64_t tpx_launch_count(void);
int tpx_profile_begin(void);
int tpx_profile_end(float* ms_by_class, int64_t* launches_by_class);

/* ------------------------------------------------------------------------------------------------------------
 * DiT  — models/dit_crossattn.py:111-213 (class DiT), constructor kwargs as in configs/inference_dit.yml:52-62
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct tpx_dit tpx_dit;
typedef struct tpx_dit_config {
    int32_t seq_length;         /* N   (2048) */
    int32_t in_channels;        /* 68  */
    int32_t out_channels;       /* 136 = 2*in (learn_sigma) */
    int32_t condition_channels; /* 768 */
    int32_t hidden_size;        /* 1152 */
    int32_t depth;              /* 28 */
    int32_t num_heads;          /* 16 */
    int32_t mlp_hidden;         /* 4608 */
} tpx_dit_config;

/* DiT.__init__ (dit_crossattn.py:115-156): allocates the packed fp16 parameter store on the current device. */
int tpx_dit_create(const tpx_dit_config* cfg, tpx_dit** out);
void tpx_dit_destroy(tpx_dit* h);
/* nn.Module.load_state_dict (inference.py:262, sd['ema']): one call per reference key
 * ("blocks.3.crossattn.to_q.weight", "final_layer.linear.bias", "null_cond_embedding", ...).  `dev_ptr` is a
 * contiguous device tensor of dtype TPX_DTYPE_*; shape is checked against the module tree.  Unknown key -> TPX_ERR_KEY. */
int tpx_dit_set_weight(tpx_dit* h, const char* ref_key, const void* dev_ptr, int dtype, const int64_t* shape, int ndim, void* stream);
/* Read a parameter back from the packed store (fp16 values, written as `dtype`) into dst_dev (same element count as the key's
 * reference shape).  Lets the host mirror drop its copy of the checkpoint after ingestion (SURVEY.md §8f-4) and still answer
 * state_dict() / move between devices. */
int tpx_dit_get_weight(tpx_dit* h, const char* ref_key, void* dst_dev, int dtype, void* stream);
/* Call once after the last set_weight: checks every required key arrived, derives the per-block constant of the
 * all-null cross-attention (proj(to_v(null_cond_embedding)), SURVEY §8a a8). */
int tpx_dit_finalize(tpx_dit* h, void* stream);

/* Bytes of the persistent conditioning store for `n_cross` sequences with `M` context tokens, and of the per-call
 * scratch for `n_seq` sequences (n_seq = 2*B under CFG). */
size_t tpx_dit_cond_bytes(const tpx_dit* h, int n_cross, int M);
size_t tpx_dit_workspace_bytes(const tpx_dit* h, int n_seq);
/* Hoist of MemEffCrossAttention.to_k/to_v (attention.py:106-107) for all blocks: they depend only on the context y,
 * so they are computed once per image instead of once per step.  y: device fp32 [n_cross, M, condition_channels]. */
int tpx_dit_set_cond(tpx_dit* h, const float* y_dev, int n_cross, int M, void* cond_ws, size_t cond_bytes, void* stream);

/* DiT.forward (dit_crossattn.py:184-202) when use_cfg == 0, DiT.forward_with_cfg (:204-213) when use_cfg != 0.
 *   x   device fp32 [B, N, in_channels];  t  device int64 [B] (ORIGINAL-schedule timesteps);
 *   out device fp16 [B, N, out_channels].
 * use_cfg == 0 : B sequences, all attend to the stored context (set_cond n_cross == B).
 * use_cfg == 1 : batch [x;x], context [y;null]; the null half uses the derived constant (n_cross == B).
 * use_cfg == 2 : same, but the null half runs real cross-attention (set_cond was given [y;null], n_cross == 2B);
 *                exists so tests can check the constant identity on the device. */
int tpx_dit_forward(tpx_dit* h, const float* x_dev, const int64_t* t_dev, int B, int use_cfg, float cfg_scale, void* out_f16_dev, void* ws,
                    size_t ws_bytes, void* stream);
/* Hoist of TimestepEmbedder (models/utils.py:27-64) and of every adaLN_modulation Linear (dit_crossattn.py:40-43,54 and :66-69,75)
 * out of the sampling loop: they depend only on the timestep, and a sampling loop visits a fixed list of them
 * (SpacedDiffusion.timestep_map, respace.py:73-87; gaussian_diffusion.py:674-685 feeds the same t to the whole batch).
 * tpx_dit_set_timesteps computes the [K, 28*9*D + 2*D] fp16 modulation rows of K original-schedule timesteps (host int64 array)
 * into caller memory `ts_ws` (256-B aligned, tpx_dit_timesteps_bytes(h, K) bytes, must stay alive and untouched while used) with
 * the same kernels and the same per-element arithmetic a forward uses, 8 timesteps per pass over the 669 MB of adaLN weights.
 * tpx_dit_forward_step is tpx_dit_forward for a batch whose B samples all sit at timestep `t`: it reads the row of `t` from that
 * table instead of running the timestep MLP and the adaLN pass (results are bit-identical to tpx_dit_forward).  `t` must be one
 * of the K values (TPX_ERR_STATE otherwise); loading a weight invalidates the table. */
size_t tpx_dit_timesteps_bytes(const tpx_dit* h, int K);
int tpx_dit_set_timesteps(tpx_dit* h, const int64_t* t_host, int K, void* ts_ws, size_t ts_bytes, void* stream);
int tpx_dit_forward_step(tpx_dit* h, const float* x_dev, int64_t t, int B, int use_cfg, float cfg_scale, void* out_f16_dev, void* ws, size_t ws_bytes,
                         void* stream);
/* Debug / parity: copy the fp32 residual stream [n_seq, N, hidden] left in `ws` by the last forward. */
int tpx_dit_debug_residual(const tpx_dit* h, const void* ws, int n_seq, float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Sampler update — models/diffusion/gaussian_diffusion.py:255-338 (p_mean_variance, LEARNED_RANGE variance),
 * :531-578 (ddim_sample), :397-440 (p_sample).  Coefficients are the float64 tables evaluated at the step and
 * rounded to fp32 exactly like _extract_into_tensor (:880-892); the host mirror computes them.
 * pred_xstart = sqrt_ab * x - sqrt_1mab * model_out (one rounding per op): with (sqrt(ab), sqrt(1-ab)) this is VELOCITY (:340-344, the
 * released model), with (sqrt(1/ab), sqrt(1/ab-1)) EPSILON (:346-351), with (0, -1) START_X (:319-320); clip != 0 clamps it to [-1, 1]
 * (process_xstart, :310-315).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct tpx_sampler_coefs {
    float sqrt_ab, sqrt_1mab, sqrt_recip_ab, sqrt_recipm1_ab;
    float c_x0, c_eps, sigma, nonzero; /* DDIM: sqrt(ab_prev), sqrt(1-ab_prev-sigma^2), sigma, (t != 0) */
    float coef1, coef2, min_log, max_log; /* DDPM: posterior mean coefficients, log-variance range */
    int32_t clip;
} tpx_sampler_coefs;
/* x, noise (may be NULL), x_prev, pred_x0: device fp32 [n]; model_out: device [n/C tokens, 2C] fp16 or fp32. */
int tpx_sampler_step(int ddim, const float* x_dev, const void* model_out_dev, int model_out_dtype, const float* noise_dev, int64_t n, int C,
                     const tpx_sampler_coefs* k, float* x_prev_dev, float* pred_x0_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Sample -> decode glue (SURVEY §8a a13 / a15) — inference.py:328-332,343-348 ; app.py:119-123,134-139
 * ---------------------------------------------------------------------------------------------------------- */
/* a13: sample device fp32 [T, C] (T = batch * num_prims, C = 68).  With per-channel statistics (mean/std device fp32 [C]):
 * v = sample * inv_nf * std + mean, one rounding per op as the reference's eager CUDA ops (x / python_float = x * fp32(1/nf));
 * without (mean == std == NULL): srt = sample[:, 0:4], z = sample[:, 4:] * inv_nf (inference.py:337).
 * Outputs: srt device fp32 [T, 4] = (scale, xyz), z device fp32 [T, C-4] = the [T,1,4,4,4] latents VAE.decode takes. */
int tpx_latent_split(const float* sample_dev, const float* mean_dev, const float* std_dev, float inv_nf, int64_t T, int C, float* srt_dev,
                     float* z_dev, void* stream);
/* a15: decoded device [T, F] (F = 6 * vox, NCDHW per primitive = channel-major; dtype fp32 or fp16) -> out device fp32 [T, 4 + F] =
 * [srt | sdf/5 | (rgb+1)/2 | (mat+1)/2], the PrimSDF / ray-marcher layout (models/primsdf.py:28-33).  srt_fix != 0 applies
 * srt[:, 0] = srt[:, 0] / 10 + 0.05 (checkpoints without per-channel statistics, inference.py:343-344). */
int tpx_primvolume_pack(const float* srt_dev, const void* decoded_dev, int decoded_dtype, int64_t T, int F, int vox, int srt_fix, float* out_dev,
                        void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * VAE decoder — models/vae3d_dib.py:391-440 (class VAE), :330-387 (Decoder)
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct tpx_vae tpx_vae;
typedef struct tpx_vae_config {
    int32_t latent_channels; /* 1 */
    int32_t out_channels;    /* 6 */
    int32_t ch_mid;          /* up_channels[0] = 256 */
    int32_t ch_out;          /* up_channels[1] = 32 */
    int32_t attn_heads;      /* 8 */
} tpx_vae_config;
int tpx_vae_create(const tpx_vae_config* cfg, tpx_vae** out);
void tpx_vae_destroy(tpx_vae* h);
/* load_state_dict(sd['model_state_dict']) (inference.py:258): decoder.* / post_quant_conv.* keys are consumed,
 * encoder.* / quant_conv.* keys are accepted and ignored (return 1). */
int tpx_vae_set_weight(tpx_vae* h, const char* ref_key, const void* dev_ptr, int dtype, const int64_t* shape, int ndim, void* stream);
int tpx_vae_finalize(tpx_vae* h, void* stream);
size_t tpx_vae_workspace_bytes(const tpx_vae* h, int P);
/* VAE.decode (vae3d_dib.py:437-440): z device [P,1,4,4,4] (dtype z_dtype) -> out device [P,6,8,8,8] (dtype out_dtype). */
int tpx_vae_decode(tpx_vae* h, const void* z_dev, int z_dtype, void* out_dev, int out_dtype, int P, void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * VAE encoder — models/vae3d_dib.py:270-327 (Encoder), :428-435 (quant_conv, VAE.encode), :50-60 (DiagonalGaussianDistribution).
 * A handle of its own: the decoder handle, its workspace and its key contract are independent of it.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct tpx_vae_encoder tpx_vae_encoder;
typedef struct tpx_vae_encoder_config {
    int32_t in_channels;     /* 6 (1..16) */
    int32_t latent_channels; /* 1 */
    int32_t ch0;             /* down_channels[0] = 32 */
    int32_t ch1;             /* down_channels[1] = 256 */
    int32_t attn_heads;      /* 8 (head dim 32) */
} tpx_vae_encoder_config;
/* Encoder.__init__ + quant_conv (vae3d_dib.py:284-307, 428) for the released layout only; anything else -> TPX_ERR_SHAPE. */
int tpx_vae_encoder_create(const tpx_vae_encoder_config* cfg, tpx_vae_encoder** out);
void tpx_vae_encoder_destroy(tpx_vae_encoder* h);
/* load_state_dict(sd['model_state_dict']): encoder.* / quant_conv.* keys are consumed (fp32 or fp16 sources), decoder.* /
 * post_quant_conv.* keys are accepted and ignored (return 1). */
int tpx_vae_encoder_set_weight(tpx_vae_encoder* h, const char* ref_key, const void* dev_ptr, int dtype, const int64_t* shape, int ndim, void* stream);
int tpx_vae_encoder_finalize(tpx_vae_encoder* h, void* stream);
size_t tpx_vae_encoder_workspace_bytes(const tpx_vae_encoder* h, int P);
/* VAE.encode up to the posterior's parameters (vae3d_dib.py:431-433): x device [P,in_channels,8,8,8] (dtype x_dtype) ->
 * params device [P,2*latent,4,4,4] (dtype params_dtype) = quant_conv(Encoder(x)). */
int tpx_vae_encode(tpx_vae_encoder* h, const void* x_dev, int x_dtype, void* params_dev, int params_dtype, int P, void* ws, size_t ws_bytes,
                   void* stream);
/* The same schedule stopped after stage 1 conv_in, 2 down_blocks.0 (after the stride-2 conv), 3 down_blocks.1 or 4 mid_block
 * (vae3d_dib.py:313-320): out_f16 device channels-last [P,S,S,S,C] of that activation.  Parity aid. */
int tpx_vae_encode_stage(tpx_vae_encoder* h, const void* x_dev, int x_dtype, int P, int stage, void* out_f16, void* ws, size_t ws_bytes, void* stream);
/* DiagonalGaussianDistribution.__init__ (vae3d_dib.py:51-60): params device [batch, 2*half_elems] (dtype fp32 / fp16; the mean is
 * its first half per batch row) -> logvar = clamp(second half, -30, 20), std = exp(0.5 logvar), var = exp(logvar), each device
 * [batch, half_elems] in the same dtype; deterministic != 0 gives std = var = 0. */
int tpx_vae_posterior(const void* params_dev, int dtype, int64_t batch, int64_t half_elems, int deterministic, void* logvar_dev, void* std_dev,
                      void* var_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Per-kernel entry points (unit parity tests; each is one launch of one hot-path kernel)
 * ---------------------------------------------------------------------------------------------------------- */
/* out[M,N] fp16 = act(A[M,K] W[N,K]^T + bias) ; act: 0 none (optionally * post_scale, re-rounded), 1 GELU-tanh.  tile_n: 0 = auto. */
int tpx_linear(const void* A_f16, int lda, const void* W_f16, const void* bias_f16, void* out_f16, int ldo, int M, int N, int K, int act,
               float post_scale, int tile_n, void* stream);
/* xres[M,N] fp32 += h(gate[(row/rows_per_batch)%gate_batches, :] * h(A W^T + bias))   (DiTBlock residual, dit_crossattn.py:55-57) */
int tpx_linear_gated(const void* A_f16, int lda, const void* W_f16, const void* bias_f16, const void* gate_f16, int gate_bstride, int gate_batches,
                     int rows_per_batch, float* xres, int ldx, int M, int N, int K, int tile_n, void* stream);
/* Column-split + head-split store: col -> (which = col / split_cols, head, d); row -> (b = row / n_seq_tokens, n);
 * out{which}[b, head, n, DhP] (zero padded).  post_scale applies to which == 0 (attention.py:105).  The column group
 * `transposed_which` (-1 = none) is stored transposed as [b, head, DhP, transposed_ld] (tokens contiguous): the V operand
 * layout of tpx_attention_tc. */
int tpx_linear_heads(const void* A_f16, int lda, const void* W_f16, const void* bias_f16, void* out0, void* out1, void* out2, int M, int N, int K,
                     int split_cols, int H, int Dh, int DhP, int n_seq_tokens, float post_scale, int tile_n, int transposed_which, int transposed_ld,
                     void* stream);
/* y = LN(x; eps) * h(1 + scale) + shift -> fp16   (modulate(norm(x), shift, scale), utils.py:19-20) */
int tpx_ln_modulate(float* x, int rows, int D, float eps, const void* shift_f16, const void* scale_f16, int mod_bstride, int rows_per_batch,
                    int mod_batches, void* out_f16, const void* pre_gate_f16, const void* pre_const_f16, int pre_row0, void* stream);
/* memory_efficient_attention contract (attention.py:54,109): q [B,H,Nq,DhP], k/v [B,H,Nk,DhP] -> out [B,Nq,H*Dh] */
int tpx_attention(const void* q, const void* k, const void* v, void* out, int B, int H, int Nq, int Nk, int Dh, int DhP, float scale, void* stream);
/* Same contract on the tcgen05 path (Dh == 72, the released model's head size): q,k [B,H,N,80]; vT = V transposed
 * [B,H,80,NkPad], NkPad % 8 == 0, padding rows/columns finite (row 72 is replaced on chip by ones to produce the row sums). */
int tpx_attention_tc(const void* q, const void* k, const void* vT, void* out, int B, int H, int Nq, int Nk, int NkPad, int Dh, float scale, void* stream);
/* Same launch with a timeline probe: block 0 writes (tag, clock64) pairs of its MMA thread and of one softmax thread per
 * query tile into timeline_dev (3 x 1024 int64, zero-initialised by the caller).  Tuning aid. */
int tpx_attention_tc_debug(const void* q, const void* k, const void* vT, void* out, int B, int H, int Nq, int Nk, int NkPad, int Dh, float scale,
                            int64_t* timeline_dev, void* stream);
/* Timeline probe of the tcgen05 GEMM (tuning aid, tools/gemm_timeline.py): while timeline_dev is non-null every later GEMM
 * launch makes CTA b write 16 int64 at timeline_dev[16 b ..]: clock64 stamps of its producer / MMA / epilogue roles and the
 * cycles each spent waiting on its mbarriers.  NULL switches it off (the default). */
int tpx_debug_gemm_timeline(int64_t* timeline_dev);
/* out = h(uncond + h(s * h(cond - uncond)))  over [cond; uncond] halves of n_half elements (dit_crossattn.py:210-213) */
int tpx_cfg_combine(const void* both_f16, int64_t n_half, float s, void* out_f16, void* stream);
/* GroupNorm(groups, eps, affine) [+ SiLU] on a channels-last fp16 volume [P, S3, C]  (vae3d_dib.py:109,112,131-139) */
int tpx_groupnorm_silu(const void* x_f16, const void* gamma_f16, const void* beta_f16, int P, int S3, int C, int groups, float eps, int apply_silu,
                       void* out_f16, void* stream);
/* 3x3x3 / pad 1 convolution as implicit GEMM on a channels-last fp16 volume [P,S,S,S,C] (S in {4,8});
 * W_f16 is [Cout, 27*C] with k = tap*C + c, tap = (kz*3+ky)*3+kx;  out [P,S,S,S,Cout] fp16 = (conv + bias (+ resid)) * alpha. */
int tpx_conv3d_k3(const void* x_f16, const void* W_f16, const void* bias_f16, const void* resid_f16, float alpha, void* out_f16, int P, int S, int C,
                  int Cout, void* stream);
/* Stride-2 3x3x3 / pad 1 convolution (vae3d_dib.py:168, DownBlock.downsample): x [P,8,8,8,C] -> out [P,4,4,4,Cout] fp16, W as above
 * (C = Cout = 32). */
int tpx_conv3d_k3_s2(const void* x_f16, const void* W_f16, const void* bias_f16, void* out_f16, int P, int C, int Cout, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * PrimSDF point query — models/primsdf.py:52-109 (PrimSDF.forward = prim_weight + grid_sample_feat), the consumer of
 * the decoded voxels (SURVEY.md §8f-1).  x device fp32 [n,3]; srt device fp32 [K,4] = (scale, tx, ty, tz), 16-B aligned;
 * feat device fp32 [K, dim_feat*S^3] channel-major (inference.py:347); out device fp32 [n, dim_feat]:
 * column 0 = sdf, 1..3 = rgb clipped to [0,1], 4..5 = roughness/metallic clipped.  inference != 0 applies the
 * nearest-voxel SDF approximation to points no primitive covers (primsdf.py:82-101).
 * ---------------------------------------------------------------------------------------------------------- */
int tpx_primsdf_query(const float* x_dev, const float* srt_dev, const float* feat_dev, int64_t n, int K, int S, int dim_feat, int inference,
                      float* out_dev, void* stream);
/* Grid-binned version of the same query (the survey's binned gather, models/primsdf.py:104-109 / inference.py:108-116): a 32^3
 * grid over the primitives' bounding box holds, per cell, the ascending lists of primitives whose box meets the cell and of the
 * primitives that can be the nearest centre for a point of the cell; tpx_primsdf_grid_build derives them from srt on the device
 * (rebuild whenever srt changes), tpx_primsdf_query_grid walks the lists of the point's cell.  Results are identical to
 * tpx_primsdf_query (same arithmetic in the same order); points outside the grid and over-full lists take the exhaustive loop.
 * grid_ws: 256-B aligned device memory of tpx_primsdf_grid_bytes(cap_entries) bytes (8 M entries cover the shipped 2048 boxes). */
size_t tpx_primsdf_grid_bytes(int64_t cap_entries);

/* ------------------------------------------------------------------------------------------------------------
 * Ray-march preview — RayMarcher.forward (dva/ray_marcher.py:142-229) = compute_raydirs (dva/mvp/extensions/utils/
 * utils_kernel.cu:15-55) + mvpraymarch(algo 0, usebvh "fixedorder", chlast, maxhitboxes 512, blocksize (8,16))
 * (dva/mvp/extensions/mvpraymarch/mvpraymarch_subset_kernel.h:14-101): called on every 10th denoising step and for the
 * turntable (inference.py:349-350).  One batch element per blockIdx.z; all pointers device fp32, contiguous:
 * template channels-last [N,K,S,S,S,4]; primpos [N,K,3] ALREADY divided by volradius (as the reference passes it),
 * primrot [N,K,3,3], primscale [N,K,3]; camera as convert_camera_parameters returns it (campos [N,3] in world units,
 * camrot [N,3,3], focal [N,2] = diagonal of K[:2,:2], princpt [N,2]); pixel (w,h) -> ray through (w,h); stepsize = dt / volradius.
 * rgba_out [N,H,W,4] (the reference's rayrgba; RayMarcher permutes it to [N,4,H,W]).
 * ---------------------------------------------------------------------------------------------------------- */
int tpx_raymarch_preview(const float* template_chlast, const float* primpos, const float* primrot, const float* primscale, const float* campos,
                         const float* camrot, const float* focal, const float* princpt, int N, int K, int S, int H, int W, float volradius, float stepsize,
                         float fadescale, float fadeexp, float* rgba_out, void* stream);
int tpx_primsdf_grid_build(const float* srt_dev, int K, void* grid_ws, size_t grid_bytes, void* stream);
int tpx_primsdf_query_grid(const float* x_dev, const float* srt_dev, const float* feat_dev, const void* grid_ws, size_t grid_bytes, int64_t n, int K, int S,
                           int dim_feat, int inference, float* out_dev, void* stream);

/* nn.GELU() (erf form) in place on an fp16 tensor of n elements (n % 8 == 0, 16-B aligned) — the activation of the DINOv2 MLP
 * (models/conditioner/dinov2/layers/mlp.py:33-39); the rest of that encoder (SURVEY.md §8f-2) is built from the entry points above. */
int tpx_gelu_erf(void* x_f16, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TPX_B200_H */
