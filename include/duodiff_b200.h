/* duodiff_b200 — C ABI of the B200-native DuoDiff sampling path.
 *
 * The reference (razvanmatisan/duodiff) has no FFI layer: its "operator API" for this path is the Python
 * module surface.  Each entry point below names the reference interface it replaces (file:line relative to
 * the reference root).  The Python shims in duodiff_b200/ bind these with ctypes; INTEGRATION.md shows the
 * stub a maintainer of the reference would add.
 *
 * Conventions: every function returns 0 on success or a negative ddb_status; ddb_last_error() returns a
 * thread-local message for the last failure.  All pointers named *_dev are CUDA device pointers owned by the
 * caller; the library never allocates caller-visible memory.  `stream` is a cudaStream_t passed as void*.
 * One handle = one device = one stream at a time (handles are not re-entrant; distinct handles are independent and
 * may be used from different threads and on different devices: the CUDA device that is current when a handle is
 * created must be current for every call on it -- the Python shims guarantee that).  The only process-wide state is
 * the set of measurement switches of ddb_set_option() (atomics, read at launch / graph-capture time).
 * There is no CPU fallback: on a machine without an sm_100 device every compute call fails with DDB_ERR_CUDA.
 */
#ifndef DUODIFF_B200_H
#define DUODIFF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    DDB_OK = 0,
    DDB_ERR_INVALID = -1,     /* bad argument / unsupported configuration */
    DDB_ERR_CUDA = -2,        /* CUDA runtime or driver error */
    DDB_ERR_MISSING_KEY = -3, /* a state_dict tensor required by the config was not supplied */
    DDB_ERR_SHAPE = -4        /* tensor size does not match the config */
} ddb_status;

/* UViT(**model_params) — models/uvit.py:229-247 (+ EarlyExitUViT, models/early_exit.py:206-266). */
typedef struct {
    int32_t img_size;
    int32_t patch_size;
    int32_t in_chans;
    int32_t embed_dim;            /* multiple of 256; head_dim = embed_dim / num_heads must be 64 */
    int32_t depth;                /* odd: depth/2 in-blocks + mid + depth/2 out-blocks */
    int32_t num_heads;
    int32_t mlp_hidden;           /* int(embed_dim * mlp_ratio) */
    int32_t num_classes;          /* <= 0: unconditional (extras = 1), else class-conditional (extras = 2) */
    int32_t normalize_timesteps;  /* models/uvit.py:352-353 */
    int32_t early_exit;           /* > 0: weights carry the EarlyExitUViT prefix `uvit.` + probes + heads; the value is
                                   * the probe layout (models/early_exit.py:194-204): 1 mlp_probe_per_layer
                                   * (matrix["i"]), 2 mlp_probe_per_timestep (matrix["t"], t < 1000),
                                   * 3 mlp_probe_per_layer_per_timestep (matrix["i, t"]), 4 attention_probe
                                   * (AttentionProbe per layer, num_heads = 1; scores are not sigmoids) */
    int32_t max_batch;            /* workspace is sized for this many samples */
    float ln_eps;                 /* nn.LayerNorm default 1e-5 */
} ddb_uvit_config;

/* One entry of the reference state_dict (Q16 of SURVEY.md): fp32, contiguous, on the device. */
typedef struct {
    const char* name;    /* state_dict key, e.g. "in_blocks.0.attn.qkv.weight" */
    const float* data_dev;
    int64_t numel;
} ddb_tensor;

typedef struct ddb_model ddb_model;
typedef struct ddb_sampler ddb_sampler;

const char* ddb_version(void);
const char* ddb_last_error(void);

/* Re-packs the fp32 state_dict into bf16 GEMM layouts (LayerNorm folded), allocates the workspace and encodes
 * the TMA descriptors.  Replaces: UViT.__init__ + load_state_dict + .to(device) (sampler.py:271-302). */
int ddb_model_create(const ddb_uvit_config* cfg, const ddb_tensor* tensors, int32_t n_tensors, ddb_model** out);
void ddb_model_destroy(ddb_model* m);

/* UViT.forward(x, timesteps, y) -> eps   (models/uvit.py:351-383)
 *   x_dev [B,C,H,W] f32; t_dev [B] f32 (raw timesteps); y_dev [B] i64 or NULL; eps_dev [B,C,H,W] f32. */
int ddb_uvit_forward(ddb_model* m, const float* x_dev, const float* t_dev, const int64_t* y_dev, int32_t B,
                     float* eps_dev, void* stream);

/* Same forward with a CUDA-event pair recorded on `stream` around every kernel launch; per-category device time
 * (ms) and launch counts are returned in host arrays of DDB_PROF_CATEGORIES entries, in the order
 * embed, ln_stats, gemm_qkv, attention, gemm_proj, gemm_fc1, gemm_fc2, gemm_skip, gemm_decode, conv, ee_other, ddpm,
 * tail (the sampler's fused conv + DDPM update + next-step head kernel; ddb_sampler_profile_step only).
 * ee != 0 also evaluates probes and heads (early-exit model).  Used by bench.py for the roofline figures. */
#define DDB_PROF_CATEGORIES 13
int ddb_profile_forward(ddb_model* m, const float* x_dev, const float* t_dev, const int64_t* y_dev, int32_t B,
                        float* eps_dev, int32_t ee, float* ms_host, int32_t* launches_host, void* stream);

/* EarlyExitUViT.forward (models/early_exit.py:268-320) fused with the selection of eesampler.py:62-68.
 *   eps_dev      [B,C,H,W] f32   eps of the first layer whose probe <= threshold (full model if none)
 *   exit_idx_dev [B] i32         that layer index (depth = no exit; with threshold < 0: 0 = no probe matched, like the
 *                                reference's argmax over an all-false mask)
 *   scores_dev   [depth,B] f32   classifier_outputs (NULL to skip)
 *   outputs_dev  [depth+1,B,C,H,W] f32 all head outputs + full-model output (NULL to skip)
 * mode 0 = simulate (reference semantics: every layer, probe and head is evaluated);
 * mode 1 = compact: a sample that exits at layer i takes head i's output and leaves the batch (a stayer from the end
 *          of the batch takes its place in the block input and the pending long skips), so later kernels run on fewer
 *          rows.  eps and
 *          exit_idx are bit-identical to mode 0; scores past a sample's exit are NaN ("not produced"), outputs_dev
 *          must be NULL, and the sampler's batch-mean probe log averages over the samples still in the batch. */
int ddb_ee_forward(ddb_model* m, const float* x_dev, const float* t_dev, const int64_t* y_dev, int32_t B,
                   float threshold, int32_t mode, float* eps_dev, int32_t* exit_idx_dev, float* scores_dev,
                   float* outputs_dev, void* stream);

/* One DDPM update (sampler.py:47-79 / eesampler.py:74-82 / ddpm_core.py:190-193), in place on x_dev.
 *   coef_dev [1000,4] f32 per-timestep {c0, c1, sigma, d}; mode 0: c0*(x - c1*out) + sigma*z (predict_noise),
 *   mode 1: (c1*out + c0*x) + sigma*z (predict_original / predict_previous),
 *   mode 2: (c0*(x - c1*out) + d*out) + sigma*z (DDIM, sampler.py:112-120; sigma holds the reference's sigma_t^2).
 *   z_dev: this step's noise [n] or NULL (Philox from `seed`); ignored at t == 0 (z = 0).
 *   Mode 3 (DPM-Solver++) needs the previous step's data prediction and fails with DDB_ERR_INVALID here; so do
 *   mode 4 (UniPC), which needs the previous two, and mode 5 (SDE-DPM-Solver++). */
int ddb_ddpm_step(float* x_dev, const float* model_out_dev, const float* z_dev, const float* coef_dev, int32_t t,
                  int32_t mode, uint64_t seed, int64_t n, void* stream);

/* get_samples() DDPM loop (sampler.py:128-139 incl. the model hand-off :135-136; eesampler.py:57-82).
 *   late may be NULL.  switch_t = 1000 - t_switch when the hand-off can trigger (1 <= t_switch <= 1000), else -1:
 *   `early` runs the steps with t >= switch_t, `late` the rest.
 *   ee_mode -1: plain U-ViT forward; 0 / 1: `early` is an early-exit model (simulate / compact, see ddb_ee_forward)
 *   and ee_threshold is eesampler.py's --threshold.  Any threshold is meaningful: a negative one selects layer 0's
 *   head for every sample, exactly like the reference's argmax over an all-false mask (eesampler.py:62-67).
 *   step_mode 0-2: coef_host [1000,4] as for ddb_ddpm_step.  step_mode 3: DPM-Solver++(2M), coef_host [1000,8] with
 *   rows {a, b, rho, phi, w0, w1, order, 0} (duodiff_b200.ddpm.dpm_solver_coefficients), no noise term:
 *     D_t = a*x + b*out;  D = w0*D_t + w1*D_prev (order 2) or D_t (order 1);  x' = rho*x + phi*D;  D_prev <- D_t.
 *   The sampler owns D_prev [B,C,H,W]; it persists across ddb_sampler_run_list calls (a trajectory cut into segments
 *   continues its history; a new one restarts it with its order-1 first row).  Mode 3 runs only through
 *   ddb_sampler_run_list over timesteps whose row has order 1 or 2, and is rejected with early exit (ee_mode >= 0).
 *   step_mode 4: UniPC (bh2, order 2, data prediction), coef_host [1000,12] with rows {a, b, cx, c0, c1, c2, px, p0,
 *   p1, corrector order, predictor order, 0} (duodiff_b200.ddpm.unipc_coefficients), no noise term:
 *     D = a*x + b*out;  corrector xc = x (order 0), cx*xb + c0*D + c1*D1 (order 1), ... + c2*D2 (order 2);
 *     x' = px*xc + p0*D (predictor order 1), ... + p1*D1 (order 2);  then xb <- xc, D2 <- D1, D1 <- D.
 *   The sampler owns xb, D1 and D2 [B,C,H,W]; they persist across ddb_sampler_run_list calls like D_prev of mode 3
 *   (a row with corrector order 0 starts a new history).  Mode 4 runs only through ddb_sampler_run_list over
 *   timesteps whose row has predictor order 1 or 2, and is rejected with early exit.
 *   step_mode 5: SDE-DPM-Solver++(2M) (the reverse SDE, data prediction), coef_host [1000,8] with rows {a, b, rho,
 *   phi, w0, w1, order, vs} (duodiff_b200.ddpm.sde_dpm_solver_coefficients): mode 3's update plus a noise term,
 *     x' = (rho*x + phi*D) + vs*z  where vs != 0 (every step but the final one);  D_prev <- D_t.
 *   z is the draw of the DDPM step at t: z_all_dev[t], or Philox keyed by (seed, t, global element index) as in
 *   modes 0-2, so ddb_sampler_set_noise_offset shards it exactly.  D_prev, the order check, ddb_sampler_run_list only
 *   and the rejection with early exit are as for mode 3. */
int ddb_sampler_create(ddb_model* early, ddb_model* late, int32_t switch_t, int32_t B, const float* coef_host,
                       int32_t step_mode, float ee_threshold, int32_t ee_mode, ddb_sampler** out);
void ddb_sampler_destroy(ddb_sampler* s);
/* Classifier-free guidance (U-ViT's form): every step runs the backbone on 2B rows, the conditional half with the
 * caller's labels y and the unconditional half with `null_label`, and the step tail uses
 * eps = eps_c + scale * (eps_c - eps_u) (scale 0 gives eps_c) per sample.  x, the noise keying and the traces stay
 * per sample (B rows).  Call once before the first run.  Fails with DDB_ERR_INVALID when a backbone is unconditional,
 * null_label is outside [0, num_classes) of a backbone, a backbone's max_batch < 2B, the scale is not finite, or the
 * sampler has early exit (ee_mode >= 0). */
int ddb_sampler_set_guidance(ddb_sampler* s, float scale, int64_t null_label);
/* Data-parallel sharding: `first_row` = index of this shard's first sample in the global batch (default 0).  The
 * in-kernel Philox noise is keyed by (seed, t, GLOBAL element index), so the shards of a global batch draw exactly the
 * z_t a single-GPU run of the whole batch draws: N-GPU sampling == 1-GPU sampling row for row (SURVEY.md 8e). */
int ddb_sampler_set_noise_offset(ddb_sampler* s, uint64_t first_row);
/* One eager step at timestep t on the early (late = 0) or late backbone with a CUDA-event pair around every kernel:
 * per-category device ms / launch counts like ddb_profile_forward, but of the step as the sampler runs it (fused
 * tail, early-exit kernels, DDPM update).  x_dev is updated in place. */
int ddb_sampler_profile_step(ddb_sampler* s, float* x_dev, const int64_t* y_dev, int32_t t, int32_t late,
                             float* ms_host, int32_t* launches_host, void* stream);
/* Runs steps t = t_first, t_first-1, ..., t_last in place on x_dev.
 *   z_all_dev: injected noise [1000, n] indexed by t, or NULL (Philox, `seed`).
 *   eps_trace_dev / x_trace_dev: optional [n_steps, n] per-step model output / x_{t-1} (parity tests).
 *   exit_idx_trace_dev [1000, B] i32 and score_mean_trace_dev [1000, depth] f32 are indexed by t like the
 *   reference's indices_by_timestep / error_prediction_by_timestep logs (eesampler.py:54-55,71-72); only the rows
 *   t_last..t_first are written.  In compact mode (ee_mode 1) row t of the score log holds, per layer, the mean over
 *   the samples STILL IN THE BATCH at that layer (the reference's batch mean needs the dead layers evaluated).
 *   use_graph != 0 replays one captured CUDA graph per backbone (eps/x traces must then be NULL).  The captured step
 *   only touches sampler-owned memory (x, labels and logs are staged), so caller pointers may change between calls.
 *   Fails with DDB_ERR_INVALID for a step_mode 3, 4 or 5 sampler (DPM-Solver++, UniPC and SDE-DPM-Solver++ are
 *   defined over their grid only). */
int ddb_sampler_run(ddb_sampler* s, float* x_dev, const int64_t* y_dev, const float* z_all_dev, uint64_t seed,
                    int32_t t_first, int32_t t_last, float* eps_trace_dev, float* x_trace_dev,
                    int32_t* exit_idx_trace_dev, float* score_mean_trace_dev, int32_t use_graph, void* stream);
/* Same loop over an explicit list of timesteps (host arrays of n_steps entries): the model runs at t_list[k] on the
 * late backbone when late[k] != 0, then the sampler's update rule is applied with the coefficients of t_list[k].
 * Used for the DDIM branch (sampler.py:103-126: strided schedule, hand-off `t < 1000 - t_switch` after the step) and
 * for DPM-Solver++ (step_mode 3), UniPC (step_mode 4) and SDE-DPM-Solver++ (step_mode 5) over the same grid: a
 * timestep whose table row has (predictor) order 0 fails with DDB_ERR_INVALID (so does ddb_sampler_profile_step). */
int ddb_sampler_run_list(ddb_sampler* s, float* x_dev, const int64_t* y_dev, const float* z_all_dev, uint64_t seed,
                         const int32_t* t_list_host, const uint8_t* late_host, int32_t n_steps, float* eps_trace_dev,
                         float* x_trace_dev, int32_t use_graph, void* stream);
/* ddb_sampler_run_list with the early-exit logs of ddb_sampler_run: exit_idx_trace_dev [1000, B] i32 and
 * score_mean_trace_dev [1000, depth] f32 (either may be NULL), indexed by t.  Only the rows of the timesteps in
 * t_list are written; every other row keeps the caller's contents.  Used for DDIM sampling with early exit (step_mode
 * 2, ee_mode >= 0).  Asking for a log from a sampler without early exit fails with DDB_ERR_INVALID. */
int ddb_sampler_run_list_logs(ddb_sampler* s, float* x_dev, const int64_t* y_dev, const float* z_all_dev,
                              uint64_t seed, const int32_t* t_list_host, const uint8_t* late_host, int32_t n_steps,
                              float* eps_trace_dev, float* x_trace_dev, int32_t* exit_idx_trace_dev,
                              float* score_mean_trace_dev, int32_t use_graph, void* stream);
/* samples = (x + 1) / 2, NCHW -> NHWC (sampler.py:145-146). */
int ddb_finalize_nhwc(const float* x_dev, float* out_dev, int32_t B, int32_t C, int32_t H, int32_t W, void* stream);
/* Process-wide runtime switches for A/B measurements (DESIGN.md lists them): "alt_dir", "attn_discard", "pdl",
 * "attn_token", "ee_fuse", "mlp_split", "l2_hints", ...; the measured-and-rejected kernel variants ("gemm_variant" = 1, "gemm_ts", "attn_x2",
 * "gemm_bn128", "gemm_ln_cfg") exist only in libraries built with DDB_EXPERIMENTAL=1 (ddb_version() then ends in
 * "+experimental"); selecting one in a product build fails with DDB_ERR_INVALID.  Captured step graphs are
 * re-captured after any change. */
int ddb_set_option(const char* name, int32_t value);
/* Bench-only instrumentation hooks (tools/): "attn_trace" = device buffer [items][2][8] of clock64() stamps. */
int ddb_debug_set_ptr(const char* name, void* dev_ptr);
/* number of kernels launched by this library since load (bench.py's gpu_launches) */
int64_t ddb_launch_count(void);

/* ---- KL-autoencoder decode: the step after the sampling loop for latent models (sampler.py:141-143,149-150) ----
 * FrozenAutoencoderKL(ddconfig, embed_dim, pretrained_path, scale_factor) -- models/utils/autoencoder.py:452-466;
 * only the fields the decoder reads (Decoder.__init__, :320-412).  get_autoencoder() (:503-516) uses
 * ch=128, ch_mult=[1,2,4,4], num_res_blocks=2, z_channels=4, resolution=256, out_ch=3, attn_resolutions=[]. */
typedef struct {
    int32_t ch;
    int32_t out_ch;          /* <= 8 */
    int32_t num_res_blocks;
    int32_t z_channels;      /* <= 8 */
    int32_t resolution;      /* output resolution; the latent grid is resolution / 2^(n_levels-1) (power of two >= 16) */
    int32_t embed_dim;       /* must equal z_channels (post_quant_conv is embed_dim -> z_channels) */
    int32_t n_levels;        /* len(ch_mult) <= 8 */
    int32_t ch_mult[8];      /* ch * ch_mult[i] must be a multiple of 64 */
    int32_t max_batch;       /* latents decoded per pass; larger batches are processed in chunks of this size */
    float scale_factor;      /* 0.18215 */
} ddb_ae_config;
typedef struct ddb_ae ddb_ae;
/* tensors: the FrozenAutoencoderKL state_dict (keys `post_quant_conv.*`, `decoder.*`; encoder keys are ignored here,
 * see ddb_ae_create_encoder). */
int ddb_ae_create(const ddb_ae_config* cfg, const ddb_tensor* tensors, int32_t n_tensors, ddb_ae** out);
void ddb_ae_destroy(ddb_ae* ae);
/* FrozenAutoencoderKL.decode(z) (models/utils/autoencoder.py:486-490):
 *   z_dev [B, z_channels, r, r] f32 -> img_dev [B, out_ch, resolution, resolution] f32 (NCHW, un-clipped). */
int ddb_ae_decode(ddb_ae* ae, const float* z_dev, int32_t B, float* img_dev, void* stream);
/* Same decode with CUDA events around every launch: device ms and algorithmic FLOPs per category
 * (conv3x3, upsample conv, conv1x1, attention matmuls, groupnorm, other), host arrays of DDB_AE_PROF_CATEGORIES. */
#define DDB_AE_PROF_CATEGORIES 6
int ddb_ae_profile_decode(ddb_ae* ae, const float* z_dev, int32_t B, float* img_dev, float* ms_host,
                          double* flops_host, void* stream);
/* Parity hooks: the decoder is a flat list of launches; op i leaves an NHWC bf16 (or f32) tensor behind.
 * info_out = {C, H, W, is_f32} (C == 0: nothing to dump).  decode_debug copies op_index's output of the first
 * B <= max_batch samples to dump_dev right after it ran. */
int32_t ddb_ae_num_ops(const ddb_ae* ae);
int ddb_ae_op_info(const ddb_ae* ae, int32_t i, char* name_out, int32_t name_cap, int32_t* info_out);
int ddb_ae_decode_debug(ddb_ae* ae, const float* z_dev, int32_t B, float* img_dev, int32_t op_index, void* dump_dev,
                        void* stream);

/* ---- KL-autoencoder encode: image -> latent (FrozenAutoencoderKL.encode_moments / sample / encode) ----
 * ddb_ae_create_encoder adds the Encoder + quant_conv plan to a handle made by ddb_ae_create, from the keys
 * `encoder.*` and `quant_conv.*` (other keys are ignored; a missing one gives DDB_ERR_MISSING_KEY).  in_channels
 * (<= 7) is read from encoder.conv_in.weight.  The encoder shares the decoder's workspace and plays no part in
 * decode; both plans may be used on one handle, one call at a time. */
int ddb_ae_create_encoder(ddb_ae* ae, const ddb_tensor* tensors, int32_t n_tensors);
/* encode_moments(x) = quant_conv(encoder(x)):
 *   img_dev [B, in_channels, resolution, resolution] f32 -> moments_dev [B, 2*embed_dim, r, r] f32 (mean | logvar),
 *   processed in chunks of max_batch. */
int ddb_ae_encode_moments(ddb_ae* ae, const float* img_dev, int32_t B, float* moments_dev, void* stream);
/* sample(moments) with caller-supplied standard-normal noise_dev [B, embed_dim, r, r]:
 *   z_dev = scale_factor * (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise)   [B, embed_dim, r, r] f32. */
int ddb_ae_sample(ddb_ae* ae, const float* moments_dev, const float* noise_dev, int32_t B, float* z_dev, void* stream);
/* Profile / parity hooks of the encoder plan, as for decode (same DDB_AE_PROF_CATEGORIES; the stride-2 Downsample
 * convolutions count as conv3x3, the im2col prep of conv_in as other). */
int ddb_ae_profile_encode(ddb_ae* ae, const float* img_dev, int32_t B, float* moments_dev, float* ms_host,
                          double* flops_host, void* stream);
int32_t ddb_ae_encoder_num_ops(const ddb_ae* ae);
int ddb_ae_encoder_op_info(const ddb_ae* ae, int32_t i, char* name_out, int32_t name_cap, int32_t* info_out);
int ddb_ae_encode_debug(ddb_ae* ae, const float* img_dev, int32_t B, float* moments_dev, int32_t op_index,
                        void* dump_dev, void* stream);

/* ---- single-operator entry points (used by the parity tests; same kernels as the model path) ---- */
/* out[M,N] = epi([A0|A1] W^T); bf16 row-major operands.  epi: 0 bias, 1 LN-fold, 2 LN-fold+GELU, 3 bias+residual.
 * stats_out_dev (optional, [M, N/64, 2] f32): per-row (mean, M2) of every 64-column output chunk.
 * variant 0: the model path's kernel; 2: CTA-pair (cta_group::2) 256x256 tiles; 1: single-CTA 128x256 tiles
 * (DDB_EXPERIMENTAL builds only). */
int ddb_op_gemm(const void* a0_dev, const void* a1_dev, const void* w_dev, const float* bias_dev,
                const float* colsum_dev, const float* stats_dev, int32_t nparts, int32_t ln_dim,
                const void* residual_dev, void* out_dev, float* stats_out_dev, int32_t M, int32_t N, int32_t K0,
                int32_t K1, int32_t epi, int32_t variant, void* stream);
/* softmax(q k^T / 8) v over qkv [B*L, 3*H*64] bf16 -> out [B*L, H*64] bf16 (models/uvit.py:159-164).
 * variant 0 / 2: the tcgen05/TMEM kernel of the model path (needs L = 256 + {1,2}, true for every reference config);
 * 1: generic-L mma.sync kernel, 3: two softmax threads per row (both DDB_EXPERIMENTAL builds only). */
int ddb_op_attention(const void* qkv_dev, void* out_dev, int32_t B, int32_t L, int32_t H, int32_t variant,
                     void* stream);
/* per-row (mean, M2) of x [M, D] bf16 -> stats [M,2] f32 */
int ddb_op_ln_stats(const void* x_dev, int32_t M, int32_t D, float* stats_dev, void* stream);
/* W' = bf16(W*gamma), colsum, bias' (LayerNorm folding) for W [N,K] f32 */
int ddb_op_pack_linear(const float* w_dev, const float* bias_dev, const float* gamma_dev, const float* beta_dev,
                       int32_t N, int32_t K, void* wp_dev, float* colsum_dev, float* bias_out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DUODIFF_B200_H */
