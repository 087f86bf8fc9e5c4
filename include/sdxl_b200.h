/* sdxl_b200.h — C ABI of the B200-native SDXL denoising engine (libsdxl_b200.so).
 *
 * This is the drop-in boundary for the diffusion sampling path of Gadersd/stable-diffusion-xl-burn:
 * the entry points a Rust `src/backend.rs` replacement would bind with `extern "C"` (see
 * INTEGRATION.md for the shim). Each function names the reference interface it replaces; citations
 * are file:line relative to the reference repository root.
 *
 * Conventions
 *  - Status: every function returns 0 on success, non-zero on error; `sdxl_last_error(ctx)` returns a
 *    human-readable message for the last failure on that context. No exception crosses the boundary
 *    (the reference panics on shape errors; here they are status codes).
 *  - Pointers are DEVICE pointers unless the parameter name ends in `_host` or the struct says so.
 *    Inputs are borrowed for the duration of the call; outputs are caller-allocated.
 *  - Tensors are contiguous. Public activations use the reference's layouts: NCHW for images/latents,
 *    [B,T,C] for token tensors, f16 (`uint16_t` bit pattern of IEEE binary16 == burn's `f16`) unless
 *    stated; NHWC/f32 is internal.
 *  - One sdxl_ctx per (device, stream). A ctx and the objects created from it are not thread-safe;
 *    independent ctxs are fully concurrent. All work is enqueued on the ctx stream; functions that
 *    return results to host memory synchronise that stream, all others are asynchronous.
 *  - There is NO CPU fallback: on a machine without an sm_100 GPU sdxl_ctx_create fails.
 */
#ifndef SDXL_B200_H_
#define SDXL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SDXL_API __attribute__((visibility("default")))
#else
#define SDXL_API
#endif

typedef uint16_t sdxl_half; /* IEEE binary16 bit pattern */
typedef struct sdxl_ctx sdxl_ctx;
typedef struct sdxl_unet sdxl_unet;

#define SDXL_MAX_LEVELS 8
#define SDXL_PROFILE_KINDS 24   /* entries of the per-kernel-kind arrays of the *_profile_plan entry points */

/* Mirrors DiffuserConfig (src/model/stablediffusion/mod.rs:269-278) + UNetConfig
 * (src/model/unet/mod.rs:59-69). Transformer blocks exist on levels 1 and 2 only
 * (unet/mod.rs:125,264); transformer_depths[level] is read for those levels, and
 * transformer_depths[n_levels-1] is the middle-block depth (unet/mod.rs:239). */
typedef struct sdxl_unet_cfg {
  int32_t adm_in_channels;                    /* 2816 base / 2560 refiner */
  int32_t in_channels;                        /* 4 */
  int32_t out_channels;                       /* 4 */
  int32_t model_channels;                     /* 320 base / 384 refiner */
  int32_t n_levels;                           /* len(channel_mults) */
  int32_t channel_mults[SDXL_MAX_LEVELS];     /* [1,2,4] base */
  int32_t n_head_channels;                    /* 64 (this build requires 64) */
  int32_t transformer_depths[SDXL_MAX_LEVELS];/* [_,2,10] base */
  int32_t context_dim;                        /* 2048 base / 1280 refiner */
  int32_t is_refiner;                         /* Diffuser.is_refiner: single forward, no CFG */
  int32_t n_steps;                            /* 1000 (stablediffusion/mod.rs:282) */
} sdxl_unet_cfg;

/* Mirrors Conditioning (src/model/stablediffusion/mod.rs:544-555); f16 like the reference's
 * Diffuser<LibTorch<f16>> after Conditioning::convert (src/bin/sample/main.rs:236-237).
 * n_batch images share the unconditional rows (the reference repeats them, mod.rs:535-536). */
typedef struct sdxl_conditioning {
  int32_t on_host;        /* 0: pointers are device memory, 1: host memory */
  int32_t n_batch;        /* context_full.dims()[0] */
  int32_t n_ctx;          /* 77 */
  const sdxl_half* context_full;                        /* [n_batch, n_ctx, 2048] */
  const sdxl_half* context_open_clip;                   /* [n_batch, n_ctx, 1280] */
  const sdxl_half* unconditional_context_full;          /* [n_ctx, 2048] */
  const sdxl_half* unconditional_context_open_clip;     /* [n_ctx, 1280] */
  const sdxl_half* channel_context;                     /* [n_batch, 2816] */
  const sdxl_half* channel_context_refiner;             /* [n_batch, 2560] */
  const sdxl_half* unconditional_channel_context;       /* [2816] */
  const sdxl_half* unconditional_channel_context_refiner; /* [2560] */
  int32_t resolution[2];  /* (height, width) in pixels; latent is /8 */
} sdxl_conditioning;

/* ---- context -------------------------------------------------------------------------------- */
/* Replaces the reference's fixed `LibTorchDevice::Cuda(0)` + libtorch default stream
 * (src/bin/sample/main.rs:131). cuda_stream may be NULL (the ctx creates its own). */
SDXL_API int sdxl_ctx_create(int device, void* cuda_stream, sdxl_ctx** out);
SDXL_API void sdxl_ctx_destroy(sdxl_ctx* ctx);
SDXL_API const char* sdxl_last_error(const sdxl_ctx* ctx);
SDXL_API int sdxl_ctx_synchronize(sdxl_ctx* ctx);
/* Number of this library's kernels launched on the ctx since creation (bench `gpu_launches`). */
SDXL_API uint64_t sdxl_ctx_launch_count(const sdxl_ctx* ctx);

/* ---- UNet / Diffuser ------------------------------------------------------------------------ */
/* Replaces load_diffuser_model (src/bin/sample/main.rs:35-41): builds the device-resident model from
 * a flat weight pack (format: DESIGN.md "weight pack"; tensor names = the reference's npy dump tree,
 * src/model/unet/load.rs, values f16 like the .mpk). The pack may live in host or device memory
 * (pack_on_device); the library keeps its own re-laid-out copy, the caller may free the pack. */
SDXL_API int sdxl_unet_load(sdxl_ctx* ctx, const sdxl_unet_cfg* cfg, const void* pack, size_t bytes,
                   int pack_on_device, sdxl_unet** out);
/* Multi-GPU load (SURVEY 8(b), 8(e)): prompt-sharded replicas, one process (or thread) per GPU. EVERY rank of `nccl_comm`
 * (an ncclComm_t the host application created, e.g. with ncclCommInitRank) calls this with the same cfg; only `root` passes a
 * pack (host or device), the other ranks pass pack = NULL, bytes = 0. One ncclBroadcast of the flat pack over NVLink on the
 * ctx stream (preceded by an 8-byte broadcast of its size), then the same local re-layout as sdxl_unet_load. No collective is
 * ever issued inside the sampling loop. libnccl.so.2 is resolved at first use (the copy already loaded in the process, else
 * $SDXL_B200_NCCL_LIB, else the loader path); without it the call fails with an error, the rest of the library works. */
SDXL_API int sdxl_unet_load_broadcast(sdxl_ctx* ctx, const sdxl_unet_cfg* cfg, const void* pack, size_t bytes, int pack_on_device,
                                      void* nccl_comm, int rank, int root, sdxl_unet** out);
SDXL_API void sdxl_unet_destroy(sdxl_unet* unet);
/* Step-invariant part of UNet::forward, hoisted: cross-attention K/V projections of `context`
 * (unet/mod.rs:1010-1011 for attn2) and the label-embedding MLP (unet/mod.rs:464-466).
 * context [B, n_ctx, context_dim] f16, y [B, adm_in_channels] f16. */
SDXL_API int sdxl_unet_set_conditioning(sdxl_unet* unet, int B, int n_ctx, const sdxl_half* context,
                               const sdxl_half* y);
/* == UNet::forward (src/model/unet/mod.rs:449-493) with the conditioning set above.
 * x [B,4,h,w] NCHW f16, t_host: the single timestep the reference passes as Int[1]
 * (stablediffusion/mod.rs:416), eps_out [B,4,h,w] NCHW f16 (caller-owned). */
SDXL_API int sdxl_unet_forward(sdxl_unet* unet, int B, int h, int w, const sdxl_half* x, int32_t t_host,
                      sdxl_half* eps_out);
/* Same, f32 NCHW in/out (no input/output rounding; used by the parity tests). */
SDXL_API int sdxl_unet_forward_f32(sdxl_unet* unet, int B, int h, int w, const float* x, int32_t t_host,
                          float* eps_out);

/* == Diffuser::sample_latent / sample_latent_with_inpainting / refine_latent
 * (src/model/stablediffusion/mod.rs:317-376) and the DDIM loops they call (:390-483), including
 * forward_diffuser's classifier-free guidance (:494-541; both branches are evaluated as one batched
 * forward, the combine keeps the reference's u + (c-u)*s form).
 *  step_start : 0 for sample_latent; refine_latent's step_start (e.g. 800) otherwise. When
 *               step_start > 0 `init_latent` is the latent to refine and is noised as mod.rs:363-367.
 *  init_latent: [n_batch,4,H/8,W/8] f32 NCHW. For step_start == 0 this is the initial noise
 *               (gen_noise, mod.rs:378-388); NULL => seeded Philox N(0,1) (stream seed, subsequence 0).
 *  noise      : optional injected per-call noise [n_noise,n_batch,4,H/8,W/8] f32 (refine entry noise
 *               and, for inpainting, one tensor per step in loop order); NULL => seeded Philox.
 *  inpaint_ref/inpaint_mask: both NULL, or reference latent f32 and mask bytes (1 = keep generated,
 *               mask_where semantics of mod.rs:465), each [n_batch,4,H/8,W/8].
 *  latent_out : [n_batch,4,H/8,W/8] f32 NCHW, device (or host if cond->on_host).
 * All pointer arguments live where cond->on_host says. */
SDXL_API int sdxl_sample_latent(sdxl_unet* unet, const sdxl_conditioning* cond, double guidance_scale,
                       int n_steps, int step_start, const float* init_latent, const float* noise,
                       int n_noise, uint64_t seed, const float* inpaint_ref,
                       const uint8_t* inpaint_mask, float* latent_out);

/* Step-wise control for benchmarking / external loops: */
/* prepare a sampler state for cond (uploads + hoists conditioning, allocates the latent). */
SDXL_API int sdxl_sampler_begin(sdxl_unet* unet, const sdxl_conditioning* cond, double guidance_scale);
/* == one iteration of the loop body at timestep t (alpha lookups + forward_diffuser + DDIM update)
 * on the internal latent; t_prev < 0 means alpha_prev = 1.0 (mod.rs:408-412). Asynchronous. */
SDXL_API int sdxl_sampler_step(sdxl_unet* unet, int t, int t_prev);
/* Same, but the latent comes from / goes to HOST memory inside the call (end-to-end timing):
 * latent_host [n_batch,4,h,w] f32 in, updated in place. Synchronises the stream. */
SDXL_API int sdxl_sampler_step_host(sdxl_unet* unet, int t, int t_prev, float* latent_host);
SDXL_API int sdxl_sampler_set_latent(sdxl_unet* unet, const float* latent, int on_host);
SDXL_API int sdxl_sampler_get_latent(sdxl_unet* unet, float* latent, int on_host);
/* alphas_cumprod[i] as the sampler sees it (f16-stored like the reference's .mpk, widened). */
SDXL_API double sdxl_unet_alpha(const sdxl_unet* unet, int i);
/* Algorithmic FLOPs (2*MAC over Linear/conv/attention, SURVEY 8(d) counting rule) and kernel-op count of
 * the launch plan currently built for this UNet (0 before the first forward). */
SDXL_API double sdxl_unet_plan_flops(const sdxl_unet* unet);
SDXL_API int sdxl_unet_plan_num_ops(const sdxl_unet* unet);
/* FLOPs the plan's tensor-core launches actually issue: without the K/V projections hoisted to set_conditioning, with the
 * phase-decomposed upsample convolutions at their real cost and with channel / key padding (bench: `executed_flops`). */
SDXL_API double sdxl_unet_plan_flops_executed(const sdxl_unet* unet);
/* Device time of ONE execution of the current launch plan, summed per kernel kind and measured with CUDA
 * events on the ctx stream (eager launches). Kind index: 0 implicit-GEMM (tcgen05), 1 attention, 2 GroupNorm,
 * 3 LayerNorm, 4 GEMV, 5 timestep-embedding, 6 first conv, 7 upsample copy, 8 phase-split copy, 9 f32->f16 cast.
 * All three arrays hold SDXL_PROFILE_KINDS entries (host). Used by bench.py for the per-kernel roofline. */
SDXL_API int sdxl_unet_profile_plan(sdxl_unet* unet, double* ms_by_kind_host, double* flops_by_kind_host,
                                    int* launches_by_kind_host);
/* Same measurement, one CSV row per launch (analysis aid; written to `path_host`). */
SDXL_API int sdxl_unet_profile_dump(sdxl_unet* unet, const char* path_host);
/* Diagnostics: in-kernel timeline (ns, %globaltimer) of CTA 0 of one implicit-GEMM launch on a synthetic
 * [M,K]x[K,N] problem; stamps_host[9]: see csrc/engine.cu. */
/* Diagnostics: launch ramp / drain of n_launch back-to-back launches of one Linear GEMM (see tools/igemm_gaps.py). */
SDXL_API int sdxl_dbg_igemm_gaps(sdxl_ctx* ctx, int M, int K, int N, int with_residual, int n_launch, int64_t* out_host);
SDXL_API int sdxl_dbg_igemm_timeline(sdxl_ctx* ctx, int M, int K, int N, int geglu, int with_residual,
                                     uint64_t* stamps_host);
/* Diagnostics: clock stamps of CTA 0 of one attention launch on synthetic data; stamps_host[3][256][4] (csrc/engine.cu). */
SDXL_API int sdxl_dbg_attention_timeline(sdxl_ctx* ctx, int B, int T, int S, int n_head, long long* stamps_host);
/* Diagnostics: the launch builders of the UNet / VAE / CLIP plans on caller data, for direct kernel tests. Each call builds a
 * scratch plan (weights re-laid out from a pack exactly as the model loaders do), runs it once on the ctx stream and waits.
 * Device pointers except `pack` (host, the sdxl_unet_load format). cfg_out (nullable, host): per implicit-GEMM launch
 * SDXL_DBG_CFG_FIELDS ints {pair, CM, CN, a_split_dim, BN, nstages, epi_tma, epi_box_bytes}; unused rows up to cfg_cap = -1.
 * kind (pack tensor names; shapes as the model packs):
 *   SDXL_DBG_CONV3      ResBlock 3x3 conv, "conv" [Cout,Cin,3,3] (+ "skip" [Cout,C2,1,1] fused as K columns on x2 when C2 > 0):
 *                       x f16 [B,H,W,Cin], x2 f16 [B,H,W,C2]; bias = bias_rows + bias_off with row stride bias_ld per image
 *                       (f32, the per-image time-embedding bias) or the conv bias when bias_rows is NULL; residual f32
 *                       [B*H*W, Cout] or NULL; out f32 [B*H*W, Cout] (ldo unused)
 *   SDXL_DBG_UPCONV     nearest-2x + 3x3 conv as four phase convs: x f32 [B,H,W,Cin] -> out f32 [B,2H,2W,Cout]
 *   SDXL_DBG_HEAD_HILO  output head GN(32) -> SiLU -> 3x3 conv on the hi/lo-split activation, "norm" + "conv":
 *                       x f32 [B,H,W,Cin] -> out f32 [B*H*W, ldo]
 *   SDXL_DBG_PADDED_S2  PaddedConv2d 3x3 stride 2, zero pad bottom / right: x f32 [B,H,W,Cin] -> out f32 [B,H/2,W/2,Cout]
 *   SDXL_DBG_LINEAR / _LINEAR_F16 / _GEGLU   PlanBuilder::linear, "lin" [Cin,Cout] + bias: x f16 [W, Cin] (B = H = 1),
 *                       out [W, ldo] f32 / f16 / f16 GEGLU (Cout = fused 2*n_out); residual f32 [W, ldo] or NULL */
#define SDXL_DBG_CFG_FIELDS 8
#define SDXL_DBG_CONV3 0
#define SDXL_DBG_UPCONV 1
#define SDXL_DBG_HEAD_HILO 2
#define SDXL_DBG_PADDED_S2 3
#define SDXL_DBG_LINEAR 4
#define SDXL_DBG_LINEAR_F16 5
#define SDXL_DBG_GEGLU 6
SDXL_API int sdxl_dbg_plan_gemm(sdxl_ctx* ctx, int kind, const void* pack_host, size_t pack_bytes, int B, int H, int W, int Cin,
                                int Cout, int C2, const void* x, const void* x2, const float* bias_rows, int bias_ld, int bias_off,
                                const float* residual, void* out, int ldo, int32_t* cfg_out_host, int cfg_cap);
/* GroupNorm(32) as the ResBlocks and the head record it: "norm" [C1+C2]; x1 f32 [B,HW,C1], x2 (nullable) [B,HW,C2]; y f16
 * [B,HW,C1+C2]; raw (nullable) f16(cat(x1,x2)); y_lo (nullable) f16(t - y), the rounding residue of y. */
SDXL_API int sdxl_dbg_plan_group_norm(sdxl_ctx* ctx, const void* pack_host, size_t pack_bytes, const float* x1, int C1,
                                      const float* x2, int C2, int B, int HW, int silu, sdxl_half* y, sdxl_half* raw,
                                      sdxl_half* y_lo);
/* Attention on column windows as the plans record it: q at columns q_col0.. of [B*T, q_pitch]; k / v at k_col0 / v_col0 of one
 * [B*S, kv_pitch] matrix; out [B*T, ldo]; head dim 64. small != 0: the short-sequence kernel (additive f16 mask [T,S] or NULL,
 * causal), else the tensor-core kernel (mask / causal ignored). */
SDXL_API int sdxl_dbg_plan_attention(sdxl_ctx* ctx, int small, const sdxl_half* q, int q_pitch, int q_col0, const sdxl_half* kv,
                                     int kv_pitch, int k_col0, int v_col0, int B, int T, int S, int n_head, const sdxl_half* mask,
                                     int causal, sdxl_half* out, int ldo);
/* The VAE's single-head attention of one image: q, k, v f16 [T,C] -> scores f32 [T,T] = q k^T, probs f16 [T,T] =
 * softmax(scores / sqrt(C)), vT f16 [C,T], out f16 [T,C] = probs v. T, C multiples of 64. */
SDXL_API int sdxl_dbg_plan_vae_attention(sdxl_ctx* ctx, const sdxl_half* q, const sdxl_half* k, const sdxl_half* v, int T, int C,
                                         float* scores, sdxl_half* probs, sdxl_half* vT, sdxl_half* out, int32_t* cfg_out_host,
                                         int cfg_cap);
/* seeded N(0,1) exactly as the sampler generates it (device out). */
SDXL_API int sdxl_randn(sdxl_ctx* ctx, float* out, size_t n, uint64_t seed, uint64_t subsequence);

/* ---- operator level (== the burn ops / Backend hooks the hot path is built from) ------------ */
/* == Backend::qkv_attention (src/backend.rs:4-10, libtorch impl :32-79, generic :88-128).
 * q [B,T,C], k/v [B,S,C] f16, C = n_head*64, out [B,T,C] f16. mask: NULL (UNet, unet/mod.rs:1017: tensor-core
 * flash kernel) or an additive f16 [T,S] matrix such as attn_decoder_mask (text encoders, clip/mod.rs:88: short
 * sequences, CUDA-core kernel). The VAE's single-head d=512 call (autoencoder/mod.rs:572) is served inside
 * sdxl_vae_decode_latent, not here. */
SDXL_API int sdxl_qkv_attention(sdxl_ctx* ctx, const sdxl_half* q, const sdxl_half* k, const sdxl_half* v,
                       const sdxl_half* mask, int B, int T, int S, int C, int n_head, sdxl_half* out);
/* == nn::Linear::forward: x [M,K] f16, w [K,N] f16 ([in,out], python/save.py:20-25), bias [N] f16 or
 * NULL, residual [M,N] f32 or NULL; out f32 [M,N] (out_f16 = 0) or f16. geglu != 0 => N is the fused
 * 2*n_out projection and out is [M,N/2] f16 = h[:, :N/2] * gelu_erf(h[:, N/2:]) (unet/mod.rs:942-956). */
SDXL_API int sdxl_op_linear(sdxl_ctx* ctx, const sdxl_half* x, const sdxl_half* w, const sdxl_half* bias,
                   const float* residual, int M, int K, int N, int geglu, int out_f16, void* out);
/* == nn::conv::Conv2d::forward on NHWC data: x [B,H,W,Cin] f32, w OIHW f16 (python/save.py:56-72),
 * bias [Cout] f16 or NULL; ksize 1|3 (pad = ksize/2), stride 1|2 (Downsample, unet/mod.rs:760-774),
 * upsample != 0 => nearest-2x first (Upsample::forward, unet/mod.rs:742-751). out f32 NHWC. */
SDXL_API int sdxl_op_conv2d(sdxl_ctx* ctx, const float* x, const sdxl_half* w, const sdxl_half* bias, int B, int H,
                   int W, int Cin, int Cout, int ksize, int stride, int upsample, float* out);
/* == GroupNorm::forward (+ optional SILU::forward) on NHWC f32 [B,HW,C] (groupnorm/mod.rs:52-82,
 * silu.rs:14-16); x2 (nullable) is channel-concatenated after x1 (Tensor::cat, unet/mod.rs:484).
 * out f16 [B,HW,C1+C2]. */
SDXL_API int sdxl_op_group_norm(sdxl_ctx* ctx, const float* x1, int C1, const float* x2, int C2, int B, int HW,
                       int n_group, const float* gamma, const float* beta, float eps, int silu,
                       sdxl_half* out);
/* == LayerNorm::forward (layernorm/mod.rs:34-49): x [rows,C] f32 -> f16. */
SDXL_API int sdxl_op_layer_norm(sdxl_ctx* ctx, const float* x, const float* gamma, const float* beta, float eps,
                       int rows, int C, sdxl_half* out);
/* == timestep_embedding (unet/mod.rs:21-39): t_host[n] ints -> out [n,dim] f32 (cos half, sin half). */
SDXL_API int sdxl_op_timestep_embedding(sdxl_ctx* ctx, const int32_t* t_host, int n, int dim, int max_period,
                               float* out);

/* ------------------------------------------------------------------------------------------------
 * Latent decoder (SURVEY.md §8(f) rank 1): replaces LatentDecoder::{decode_latent, latent_to_image}
 * (reference src/model/stablediffusion/mod.rs:199-237, 263-266) over Autoencoder::decode_latent and Decoder::forward
 * (src/model/autoencoder/mod.rs:66-69, 193-216). The reference hard-codes the layer widths
 * (AutoencoderConfig::init, autoencoder/mod.rs:28-45); they are parameters here only so that tests can run a
 * small instance. Weight names follow the reference's loader (autoencoder/load.rs): post_quant_conv,
 * decoder/conv_in, decoder/mid/{block_1,attn,block_2}, decoder/blocks/<i>/{res1,res2,res3,upsampler},
 * decoder/norm_out, decoder/conv_out; conv weights OIHW f16, biases / norm affine f16.
 * ------------------------------------------------------------------------------------------------ */
typedef struct sdxl_vae sdxl_vae;
typedef struct sdxl_vae_cfg {
  int32_t latent_channels;              /* 4 */
  int32_t n_blocks;                     /* 4 */
  int32_t block_in[SDXL_MAX_LEVELS];    /* 512, 512, 512, 256  (DecoderConfig channels, autoencoder/mod.rs:33) */
  int32_t block_out[SDXL_MAX_LEVELS];   /* 512, 512, 256, 128 */
  int32_t n_group;                      /* 32 */
  double scale_factor;                  /* 0.13025 for SDXL (stablediffusion/load.rs:78) */
  /* encoder half (EncoderConfig, autoencoder/mod.rs:30-31); n_enc_blocks = 0: decoder only, encoder tensors not read */
  int32_t n_enc_blocks;                 /* 4 */
  int32_t enc_in[SDXL_MAX_LEVELS];      /* 128, 128, 256, 512 */
  int32_t enc_out[SDXL_MAX_LEVELS];     /* 128, 256, 512, 512 */
  int32_t enc_z_channels;               /* 8 (mean + logvar); the first latent_channels are kept (autoencoder/mod.rs:62) */
} sdxl_vae_cfg;

/* replaces load_latent_decoder (stablediffusion/load.rs:70-84): same flat pack container as sdxl_unet_load. */
SDXL_API int sdxl_vae_load(sdxl_ctx* ctx, const sdxl_vae_cfg* cfg, const void* pack, size_t bytes, int pack_on_device,
                           sdxl_vae** out);
SDXL_API void sdxl_vae_destroy(sdxl_vae* vae);
/* == LatentDecoder::decode_latent (stablediffusion/mod.rs:263-266): latent f32 [B,C,h,w] NCHW -> image f32
 * [B,3,8h,8w] NCHW (nominally in [-1,1]). `on_host` != 0: both pointers are host memory. h*w must be a multiple of 64. */
SDXL_API int sdxl_vae_decode_latent(sdxl_vae* vae, int B, int h, int w, const float* latent, int on_host, float* image_out);
/* == LatentDecoder::latent_to_image (stablediffusion/mod.rs:200-237): RawImages buffer, u8 [B, 8h, 8w, 3],
 * value = trunc(clamp(((x + 1) / 2) * 255, 0, 255)). */
SDXL_API int sdxl_vae_latent_to_image(sdxl_vae* vae, int B, int h, int w, const float* latent, int on_host, uint8_t* rgb_out);
/* == LatentDecoder::encode_image (stablediffusion/mod.rs:258-261) over Autoencoder::encode_image (autoencoder/mod.rs:58-64):
 * image f32 [B,3,H,W] NCHW in [-1,1] -> latent f32 [B,latent_channels,H/8,W/8] (mean channels of quant_conv, times
 * scale_factor; no sampling, like the reference). Encoder weights: encoder/conv_in, encoder/blocks/<i>/{res1,res2,
 * downsampler/conv}, encoder/mid/{block_1,attn,block_2}, encoder/norm_out, encoder/conv_out, quant_conv
 * (autoencoder/load.rs:82-116). (H/8)*(W/8) must be a multiple of 64. */
SDXL_API int sdxl_vae_encode_image(sdxl_vae* vae, int B, int H, int W, const float* image, int on_host, float* latent_out);
/* == LatentDecoder::image_to_latent (stablediffusion/mod.rs:239-256): RawImages u8 [B,H,W,3] -> latent. */
SDXL_API int sdxl_vae_image_to_latent(sdxl_vae* vae, int B, int H, int W, const uint8_t* rgb, int on_host, float* latent_out);
SDXL_API double sdxl_vae_encode_plan_flops(const sdxl_vae* vae);
/* algorithmic FLOPs (2*MAC over conv / linear / QK^T / PV) of the current decode plan; per-kind CUDA-event profile and
 * per-op CSV as for the UNet plan. */
SDXL_API double sdxl_vae_plan_flops(const sdxl_vae* vae);
SDXL_API int sdxl_vae_profile_plan(sdxl_vae* vae, double* ms_by_kind, double* flops_by_kind, int* launches_by_kind);
SDXL_API int sdxl_vae_profile_dump(sdxl_vae* vae, const char* path);

/* ------------------------------------------------------------------------------------------------
 * BPE tokenizers of the Embedder (SURVEY.md §8(f) rank 2). CPU host code, no device work, no sdxl_ctx.
 * Replaces ClipTokenizer (reference src/token/clip.rs:80-230), OpenClipTokenizer (src/token/open_clip.rs:71-221) and
 * tokenize_text (src/model/stablediffusion/mod.rs:778-793). The vocabulary files are the reference's own
 * (tokenizer/clip/bpe_simple_vocab_16e6.txt; tokenizer/open_clip/{merges,vocab}.txt), passed by path. Token ids are
 * bit-exact with the reference (known-answer vector src/token/clip.rs:232-249). Errors: non-zero status,
 * text in sdxl_tokenizer_last_error() (thread-local); where the reference would panic (piece not in the vocabulary)
 * an error is returned instead.
 * ------------------------------------------------------------------------------------------------ */
typedef struct sdxl_tokenizer sdxl_tokenizer;
SDXL_API const char* sdxl_tokenizer_last_error(void);
/* == ClipTokenizer::new (clip.rs:91-122); pads with <|endoftext|> (49407) */
SDXL_API int sdxl_tokenizer_create_clip(const char* merges_path, sdxl_tokenizer** out);
/* == OpenClipTokenizer::new (open_clip.rs:82-113); pads with 0 */
SDXL_API int sdxl_tokenizer_create_open_clip(const char* merges_path, const char* vocab_path, sdxl_tokenizer** out);
SDXL_API void sdxl_tokenizer_destroy(sdxl_tokenizer* tok);
/* == Tokenizer::encode(text, add_sot, add_eot) (clip.rs:181-205). ids_out may be NULL to query *n_out. */
SDXL_API int sdxl_tokenizer_encode(const sdxl_tokenizer* tok, const char* text_utf8, int add_sot, int add_eot,
                                   uint32_t* ids_out, int capacity, int* n_out);
/* == Tokenizer::decode (clip.rs:207-213); NUL-terminated UTF-8, *n_out = length without the NUL. */
SDXL_API int sdxl_tokenizer_decode(const sdxl_tokenizer* tok, const uint32_t* ids, int n, char* out, int capacity, int* n_out);
/* == tokenize_text (stablediffusion/mod.rs:778-793): encode(text, true, true) resized to seq_len with the padding token. */
SDXL_API int sdxl_tokenize_text(const sdxl_tokenizer* tok, const char* text_utf8, int seq_len, int32_t* tokens_out);
/* start_of_text_token / end_of_text_token / padding_token (clip.rs:215-229) */
SDXL_API int sdxl_tokenizer_special(const sdxl_tokenizer* tok, uint32_t* sot, uint32_t* eot, uint32_t* pad);

/* ------------------------------------------------------------------------------------------------
 * Text encoders of the Embedder (SURVEY.md §8(f) rank 2): replaces CLIP::{forward_hidden, forward_hidden_pooled}
 * (reference src/model/clip/mod.rs:82-147) for both CLIP-L and OpenCLIP-bigG. Weight names follow
 * load_clip_text_transformer (src/model/clip/load.rs:79-115): token_embedding/weight [n_vocab,n_state],
 * position_embedding/weight [n_ctx,n_state], blocks/<i>/{attn_ln,mlp_ln}/{weight,bias},
 * blocks/<i>/attn/{query,key,value,out}/{weight [in,out],bias}, blocks/<i>/mlp/{fc1,fc2}/{weight,bias},
 * layer_norm/{weight,bias}, text_projection [n_state,embed_dim] (optional); all f16 in the pack.
 * ------------------------------------------------------------------------------------------------ */
typedef struct sdxl_clip sdxl_clip;
typedef struct sdxl_clip_cfg {          /* == CLIPConfig (clip/mod.rs:18-26) */
  int32_t n_vocab;                      /* 49408 */
  int32_t n_state;                      /* 768 CLIP-L, 1280 OpenCLIP-bigG */
  int32_t embed_dim;                    /* 768 / 1280 */
  int32_t n_head;                       /* 12 / 20 (head dim 64) */
  int32_t n_ctx;                        /* 77 */
  int32_t n_layer;                      /* 12 / 32 */
  int32_t quick_gelu;                   /* 1 CLIP-L (QuickGELU), 0 OpenCLIP (erf GELU) */
} sdxl_clip_cfg;
SDXL_API int sdxl_clip_load(sdxl_ctx* ctx, const sdxl_clip_cfg* cfg, const void* pack, size_t bytes, int pack_on_device,
                            sdxl_clip** out);
SDXL_API void sdxl_clip_destroy(sdxl_clip* clip);
/* == CLIP::forward_hidden(tokens [B,n_ctx], hidden_idx): the stream after blocks[0..hidden_idx], f32 [B,n_ctx,n_state].
 * tokens are host int32 (tokenize_text output); the causal mask is applied as attn_decoder_mask does (backend.rs:21). */
SDXL_API int sdxl_clip_forward_hidden(sdxl_clip* clip, int B, const int32_t* tokens_host, int hidden_idx, float* hidden_out,
                                      int out_on_host);
/* == CLIP::forward_hidden_pooled: hidden as above plus pooled [B,embed_dim] = layer_norm(x_final)[b, argmax(tokens[b])] @ text_projection */
SDXL_API int sdxl_clip_forward_hidden_pooled(sdxl_clip* clip, int B, const int32_t* tokens_host, int hidden_idx,
                                             float* hidden_out, float* pooled_out, int out_on_host);
SDXL_API double sdxl_clip_plan_flops(const sdxl_clip* clip);

/* ---- `sample` front-end helpers --------------------------------------------------------------------- */
/* Inpainting mask from a crop window in pixels (src/bin/sample/main.rs:144-190): latent coordinates = pixel / (img_h / lat_h),
 * ones inside the window, zero outside, inverted by crop_out; mask = 1 keeps the generated latent. Negative bound = not given
 * (0 / image extent). Output: host uint8 [n_channels, lat_h, lat_w] (the [1,4,h,w] Bool tensor of the reference). */
SDXL_API int sdxl_make_inpaint_mask(int img_w, int img_h, int lat_w, int lat_h, int crop_left, int crop_right, int crop_top,
                                    int crop_bottom, int crop_out, int n_channels, uint8_t* mask_out_host);

/* ---- burn record (.mpk) helper ----------------------------------------------------------------------- */
/* The reference ships weights as burn 0.13 NamedMpkFileRecorder<HalfPrecisionSettings> records (src/bin/convert/main.rs:65-70,
 * loaded at src/bin/sample/main.rs:28-51): MessagePack, tensors as {"value": [f16 bit patterns as msgpack uints], "shape": [..]}.
 * sdxl_b200/burn_record.py walks the tree; these decode / encode the value arrays (host memory, no CUDA). */
SDXL_API int sdxl_mpk_decode_u16(const uint8_t* buf, size_t len, size_t count, uint16_t* out, size_t* consumed);
SDXL_API size_t sdxl_mpk_encode_u16(const uint16_t* in, size_t count, uint8_t* out);

#ifdef __cplusplus
}
#endif
#endif /* SDXL_B200_H_ */
