/*
 * panacea_b200 — C ABI of the B200-native Panacea denoising hot path.
 *
 * Drop-in boundary (SURVEY.md section 8b). The reference is pure Python with no FFI of its own; the
 * interface this library stands behind is the `nn.Module.forward` surface of
 *   sgm/modules/diffusionmodules/wrappers.py:37-70     OpenAIWrapperControlLDM3D.forward
 *   sgm/modules/diffusionmodules/controlmodel.py:86-202 ControlNet3D / ControlledUNetModel3D.forward
 *   sgm/modules/diffusionmodules/openaimodel.py:499-542 ResBlock3D._forward
 *   sgm/modules/attention.py:407-610,229-291,1064-1134  view / text / temporal attention, STT
 *   sgm/modules/diffusionmodules/sampling.py:96-133     EulerEDMSampler step
 *   sgm/modules/diffusionmodules/sampling.py:136-365    the other samplers' updates
 * and every entry point below names the reference call site it replaces. The Python host
 * (panacea_b200/sgm/...) mirrors those classes and binds these symbols with ctypes (INTEGRATION.md).
 *
 * Conventions
 *  - plain pointers + sizes only; all tensor pointers are DEVICE pointers owned by the caller;
 *  - activations are channels-last: fp32 residual stream [frames, H, Wtot, C], bf16 MMA operands;
 *    frame index = b*T + t (t fastest), Wtot = 6 views side by side (view-major along W);
 *  - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it and allocation-free
 *    (CUDA-graph capturable); a handle-free design: no hidden device state except memoised TMA maps;
 *  - return 0 on success, negative pn_status otherwise; message via pn_last_error() (thread-local);
 *  - there is NO CPU fallback anywhere: without a CUDA device every compute entry point fails.
 */
#ifndef PANACEA_B200_H
#define PANACEA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PN_ABI_VERSION 3

enum pn_status { PN_STATUS_OK = 0, PN_STATUS_INVALID = -1, PN_STATUS_CUDA = -2, PN_STATUS_UNSUPPORTED = -3 };

/* How a producer writes the A operand of the GEMM that follows it ("operand_mode" arguments below).
 *  PN_OPERAND_BF16   bf16 [rows, C]                   — the fast path (bf16 products, fp32 accumulation);
 *  PN_OPERAND_SPLIT3 bf16 [rows, 3C] = [hi | lo | hi] — parity mode: hi = bf16(v), lo = bf16(v - hi); against weights
 *                    packed [W_hi | W_hi | W_lo] per tap the same pn_gemm kernel yields fp32-class products
 *                    (hi W_hi + lo W_hi + hi W_lo), which is how the reference's fp32 math (wrappers.py:37-70 on CPU)
 *                    is matched to rtol 1e-3 / atol 1e-4;
 *  PN_OPERAND_F32    fp32 [rows, C]                   — input of a CUDA-core consumer in parity mode. */
enum pn_operand_mode { PN_OPERAND_BF16 = 0, PN_OPERAND_SPLIT3 = 1, PN_OPERAND_F32 = 2 };

const char* pn_last_error(void);
int pn_abi_version(void);

/* ------------------------------------------------------------------------------------------------
 * pn_gemm — tcgen05 GEMM / implicit-GEMM convolution (sm_100a, TMA + TMEM).
 * Replaces: nn.Linear (attention.py:94,113,220-226; openaimodel.py:939-941), nn.Conv2d 3x3 stride 1 over
 * the 6-view panorama (openaimodel.py:413,455-462,125), nn.Conv1d k=3 over frames (openaimodel.py:418,
 * 468-476), 1x1 skip / zero convs (openaimodel.py:486; controlmodel.py:81-84).
 *   out[row, n] = epi( sum_{th,tw,c} A[nb, y+th-taps_h/2, x+tw-taps_w/2, c] * B[n, (th*taps_w+tw)*C + c] )
 * with zero padding outside [0,H)x[0,W) and row = (nb*H + y)*W + x.
 * epi: + bias[n] + rowvec[(row / rows_per_group) % n_groups, n]; GEGLU (columns in blocks of 32 = 16 value
 * columns then the 16 gate columns of the same outputs -> N/2 outputs, out = value * gelu_erf(gate), attention.py:91-99); + residual[row, n] + residual2[row, n] (fp32); store fp32 or bf16.
 * ---------------------------------------------------------------------------------------------- */
typedef struct pn_gemm_args {
  const void* A;          /* bf16 [NB, H, W, C] with element strides below (C contiguous) */
  const void* B;          /* bf16 [N, taps_h*taps_w*C], K contiguous */
  void* out;              /* fp32 or bf16 [NB*H*W, ldo] */
  const float* bias;      /* [N] or NULL */
  const float* rowvec;    /* [n_groups, N] or NULL */
  const void* residual;   /* fp32 (or bf16 when residual_bf16) [NB*H*W, ldr] or NULL (may alias out when same dtype) */
  const float* residual2; /* second fp32 addend [NB*H*W, ldr2] or NULL (fp32 output only) */
  int64_t NB, H, W, C;
  int64_t a_stride_w, a_stride_h, a_stride_n; /* elements */
  int64_t ldo, ldr, ldr2;
  int64_t rowvec_ld;      /* row stride of rowvec in elements (0 = N) */
  int32_t N;
  int32_t taps_h, taps_w;
  int32_t rows_per_group, n_groups;
  int32_t out_bf16;
  int32_t geglu;
  int32_t residual_bf16;  /* the residual is bf16 (bf16 output only): the transformer blocks' bf16 token stream */
  /* LayerNorm folded into the GEMMs around the bf16 token stream (attention.py:699-701 + :726-747, norm1/2/3):
   * ln_stats_out — this GEMM (1x1, K <= 640, bf16 out) also writes, per output row, pn_gemm_ln_parts(N) partial
   *   (sum, sum of squares) pairs of the bf16 values it stores: float [rows][parts][2];
   * ln_stats_in / ln_parts_in / ln_colsum / ln_eps — (1x1, K <= 640, bf16 out, no GEGLU) A is the UN-normalised stream, B = W diag(gamma); the epilogue
   *   finishes the LayerNorm: out = rstd_m (acc - mean_m s_n) + bias_n with s_n = ln_colsum[n] = sum_k B[n,k] and the
   *   caller's bias_n = sum_k beta_k W[n,k] (+ the layer's own bias); mean/rstd over the C = K channels of row m. */
  const float* ln_stats_in;
  const float* ln_colsum;
  float* ln_stats_out;
  int32_t ln_parts_in;
  float ln_eps;
} pn_gemm_args;

int pn_gemm(const pn_gemm_args* args, void* stream);
int pn_gemm_ln_parts(int N);

/* ------------------------------------------------------------------------------------------------
 * pn_attention — tcgen05 flash attention over view-tiled tokens (head_dim 64).
 * Replaces: xformers.ops.memory_efficient_attention inside MemoryEfficientIntraViewAttention.forward
 * (attention.py:407-489) and MemoryEfficientInterViewAttentionTwo.forward (attention.py:518-610), and
 * F.scaled_dot_product_attention inside CrossAttention.forward for the 77-token text context
 * (attention.py:229-291). Query tokens are a grid [F, H, V, W] (frame, row, view, column) with token
 * stride q_ld; key/value tokens a grid [F / kv_frame_div, Hk, Vk, Wk] with stride kv_ld. Query view v
 * attends the key views kv_views[v][0 .. kv_view_count[v]) (all rows/columns of those views):
 *   intra-view : kv_views[v] = {v};   cross-view : the reference's table {5,1},{0,2},{1,3},{2,4},{3,5},{4};
 *   text       : V = Vk = 1, W = tokens per batch element, Wk = 77, kv_views[0] = {0}.
 * out[token, head*64 + d] = softmax(q k^T * scale) v, bf16, token stride out_ld.
 * ---------------------------------------------------------------------------------------------- */
typedef struct pn_attn_args {
  const void* q;   /* bf16, channel 0 of head 0 of the first query token */
  const void* k;   /* bf16, likewise for keys (may point into the same fused qkv buffer) */
  const void* v;
  void* out;       /* bf16 */
  int64_t q_ld, kv_ld, out_ld;
  int64_t F, H, V, W;
  int64_t Hk, Vk, Wk;
  int32_t kv_frame_div;
  int32_t heads, head_dim;
  int32_t kv_views[8][2];
  int32_t kv_view_count[8];
  float scale;
} pn_attn_args;

int pn_attention(const pn_attn_args* args, void* stream);

/* Temporal self-attention over T <= 16 frames per pixel (attention.py:1116-1125 -> :229-291, context=None).
 * q/k/v/out bf16 [batch, T, pixels, ld]; one (batch, pixel, head) sequence per warp (warp-level bf16 MMAs, fp32
 * softmax); ld and out_ld multiples of 8. */
int pn_attention_temporal(const void* q, const void* k, const void* v, void* out, int64_t batch, int64_t T,
                          int64_t pixels, int32_t heads, int32_t head_dim, int64_t ld, int64_t out_ld, float scale,
                          void* stream);

/* Parity-mode attention: the same geometry (pn_attn_args; q/k/v are fp32 here, strides in floats, out_ld must be
 * heads*head_dim), fp32 products / softmax / accumulation on CUDA cores, head_dim 64 or 80; `out` is written as the
 * operand of the to_out GEMM in `operand_mode`. Same reference call sites as pn_attention / pn_attention_temporal. */
int pn_attention_f32(const pn_attn_args* args, int operand_mode, void* stream);
int pn_attention_temporal_f32(const float* q, const float* k, const float* v, void* out, int64_t batch, int64_t T,
                              int64_t pixels, int32_t heads, int32_t head_dim, int64_t ld, float scale, int operand_mode,
                              void* stream);

/* ------------------------------------------------------------------------------------------------
 * Normalisation (fp32 residual stream in, bf16 MMA operand out)
 * ---------------------------------------------------------------------------------------------- */
/* GroupNorm(32, C) over (C/32, all pixels of a frame) [+ SiLU]: util.py:276-283 (eps 1e-5, ResBlock3D
 * in/out_layers, openaimodel.py:413,455) and attention.py:129-132 (eps 1e-6, STT norm*). The statistics span
 * all six views of the panorama. raw_bf16 (optional) receives a plain bf16 cast of x (input of the 1x1 skip
 * convolution, openaimodel.py:486). workspace: pn_groupnorm_workspace_floats(...) floats. */
int64_t pn_groupnorm_workspace_floats(int64_t frames, int64_t pixels, int64_t channels);
int pn_groupnorm_silu(const float* x, const float* gamma, const float* beta, void* y, void* raw,
                      float* workspace, int64_t frames, int64_t pixels, int64_t channels, float eps, int act_silu,
                      int operand_mode, void* stream);
/* GroupNorm(32, C) over (C/32, T) per pixel [+ SiLU] on x[batch, T, pixels, C]: the reference applies
 * nn.GroupNorm to the "(b h w) c t" rearrangement (openaimodel.py:509-512, 534-537). */
int pn_groupnorm_pixel_silu(const float* x, const float* gamma, const float* beta, void* y, int64_t batch,
                            int64_t frames_per_seq, int64_t pixels, int64_t channels, float eps, int act_silu,
                            int operand_mode, void* stream);
/* nn.LayerNorm(C) per token, eps 1e-5 (attention.py:699-701). x: fp32, or bf16 (x_is_bf16: the bf16 token stream the
 * fast path keeps inside a transformer block). */
int pn_layernorm(const void* x, int x_is_bf16, const float* gamma, const float* beta, void* y, int64_t rows,
                 int64_t channels, float eps, int operand_mode, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Convolutions that cannot feed a 64-wide UMMA K block, layout and sampler helpers
 * ---------------------------------------------------------------------------------------------- */
/* Direct 3x3 conv, pad 1, stride 1|2, channels-last (stem openaimodel.py:977, head :1251, BEV hint stem
 * controlmodel.py:43-59). w_packed fp32 [9][Cin][Cout_pad]; y = act(conv + bias) + addend. */
int pn_conv3x3_direct(const void* x, int x_is_bf16, const float* w_packed, const float* bias, const float* addend,
                      float* y_f32, void* y_bf16, int64_t frames, int64_t H, int64_t W, int64_t Cin, int64_t Cout,
                      int64_t Cout_pad, int stride, int act_silu, void* stream);
/* im2col for the stride-2 Downsample conv: fp32 [F,H,W,C] -> operand [F*Ho*Wo, 9 taps x C] (each tap is one operand
 * row of C channels: 9*C bf16, or 9*3C in split3 mode). pad = 1: Conv2d(3, stride 2, padding 1) of the UNet
 * (openaimodel.py:187); pad = 0: the VAE encoder's F.pad(x, (0,1,0,1)) + Conv2d(3, stride 2, padding 0) (model.py:98-113). */
int pn_im2col3x3_s2(const float* x, void* out, int64_t frames, int64_t H, int64_t W, int64_t C, int pad, int operand_mode,
                    void* stream);
/* F.interpolate(scale_factor=2, mode="nearest") of Upsample (openaimodel.py:133-140), fp32 -> operand. */
int pn_upsample2x(const float* x, void* y, int64_t frames, int64_t H, int64_t W, int64_t C, int operand_mode, void* stream);
/* out = cat([h, skip + ctrl], channel) — decoder skip join (controlmodel.py:193-195); ctrl may be NULL. */
int pn_concat_add(const float* h, const float* skip, const float* ctrl, float* out, int64_t rows, int64_t C1,
                  int64_t C2, void* stream);
int pn_add_inplace(float* x, const float* y, int64_t n, void* stream);      /* h += control.pop() (controlmodel.py:192) */
/* fp32 [rows, C] -> operand (bf16 or split3). */
int pn_cast_operand(const float* x, void* y, int64_t rows, int64_t C, int operand_mode, void* stream);
/* Parity-mode GEGLU (attention.py:97-99, exact erf GELU) on the fp32 output of the ff.net.0 GEMM whose columns are in
 * pn_gemm's GEGLU packing (blocks of 32 = 16 value + 16 gate columns): in fp32 [rows, 2*inner] -> operand [rows, inner]. */
int pn_geglu_operand(const float* in, void* y, int64_t rows, int64_t inner, int operand_mode, void* stream);
/* in[batch, A, first B of in_ld columns] -> out[batch, B, ld] at column offset off: NCHW <-> channels-last at the module
 * boundary (also performs the channel concat of wrappers.py:41, and drops the padding columns of the out-head GEMM). */
int pn_transpose_f32(const float* in, float* out, int64_t batch, int64_t A, int64_t B, int64_t in_ld, int64_t out_ld,
                     int64_t out_off, void* stream);
/* util.py:224-248 timestep_embedding (cos | sin halves). freqs: optional fp32 [dim/2] frequency table computed by the
 * host with the reference's expression (bit-identical arguments t*f); NULL = computed in the kernel. */
int pn_timestep_embedding(const int64_t* t, float* out, int64_t n, int64_t dim, const float* freqs, void* stream);
/* y = act_out(W act_in(x) + b) for M <= 32 rows: time_embed MLP and per-block emb_layers
 * (openaimodel.py:936-943, 439-445). */
int pn_linear_small(const float* x, const void* W, int w_is_f32, const float* bias, float* y, int64_t M, int64_t N,
                    int64_t K, int64_t ldy, int silu_in, int silu_out, void* stream);
/* out[r, :] = softmax(scale * in[r, :]), fp32 scores -> bf16 probabilities. With two pn_gemm calls around it this is the
 * single-head attention of the VAE mid block (reference sgm/modules/diffusionmodules/model.py:374-414, head_dim = C). */
int pn_softmax_rows(const float* in, void* out_bf16, int64_t rows, int64_t N, int64_t ld_in, int64_t ld_out, float scale,
                    void* stream);
/* Content fingerprint of a device buffer (two order-independent 64-bit sums over its 32-bit words) -> out2[2] on the
 * device. The wrapper keys its step-invariant conditioning cache (BEV hint stem, text K/V; wrappers.py:37-70 recomputes
 * them every step) on the CONTENT of c["cond_feat"] / c["crossattn"]: addresses are recycled by the allocator. */
int pn_fingerprint(const void* x, int64_t nbytes, uint64_t* out2, void* stream);
/* out[c*n + i] = x[i] * s for c < copies (prepare_sampling_loop x *= sqrt(1+sigma0^2), CFG batch doubling). */
int pn_scale_dup(const float* x, float* out, int64_t n, float s, int copies, void* stream);

/* ------------------------------------------------------------------------------------------------
 * pn_sampler_step — one fused update of the reference's samplers per network evaluation
 * (sampling.py:96-365, sampling_utils.py:27-48, denoiser.py:22-28, guiders.py:25-29), fp32, reference operation
 * order. Per element e < n:
 *   den   = CFG(net2[e], net2[n+e]) with EpsScaling applied at the evaluation point xe (x, or x_eval for the *_B modes):
 *           den_h = net_h * (-sigma_q) + xe, den = den_u + cfg_scale (den_c - den_u); net_is_denoised: den_h = net_h;
 *   mode  PN_SAMPLER_INPUT      no network output: x only receives the noise below (EDM churn before the first step);
 *         PN_SAMPLER_EULER      d = (x - den) / sigma; x += dt d  (EDM Euler dt = sigma_next - sigma_hat; Euler-ancestral
 *                               dt = sigma_down - sigma; the single-evaluation steps of Heun / DPM++ 2S a);
 *         PN_SAMPLER_HEUN_A     d = (x - den) / sigma -> d[e]; x_eval = x + dt d (x unchanged);
 *         PN_SAMPLER_HEUN_B     d' = (x_eval - den) / sigma (sigma = sigma_next); x += ((d[e] + d') / 2) dt;
 *         PN_SAMPLER_DPMPP2S_A  x_eval = m1 x - m2 den (x unchanged);
 *         PN_SAMPLER_DPMPP2S_B  x = m3 x - m4 den;
 *         PN_SAMPLER_DPMPP2M    x = m1 x - m2 (m3 den - m4 old_denoised[e]) if use_old, else x = m1 x - m2 den;
 *                               then old_denoised[e] = den;
 *         PN_SAMPLER_LMS        d = (x - den) / sigma -> d[lms_slot]; x += sum_j lms_coeff[j] d[(lms_slot - j) mod lms_ring]
 *                               for j < lms_order (newest first, summed left to right);
 *   noise (every mode but the *_A ones): x += (z * noise_mul) * noise_amp with z = noise[e] (PN_NOISE_BUFFER) or
 *         pn_philox_normal's value for (seed, draw, e) (PN_NOISE_PHILOX);
 *   x_in_next (optional, 2n): the next network input, (x_eval for the *_A modes, else the new x) * c_in_next, twice.
 * d / x_eval / old_denoised are state buffers owned by the sampler (latent-sized fp32; d holds lms_ring latents for
 * LMS); none may alias net2. */
enum pn_sampler_mode {
  PN_SAMPLER_INPUT = 0, PN_SAMPLER_EULER = 1, PN_SAMPLER_HEUN_A = 2, PN_SAMPLER_HEUN_B = 3,
  PN_SAMPLER_DPMPP2S_A = 4, PN_SAMPLER_DPMPP2S_B = 5, PN_SAMPLER_DPMPP2M = 6, PN_SAMPLER_LMS = 7
};
enum pn_noise_source { PN_NOISE_NONE = 0, PN_NOISE_PHILOX = 1, PN_NOISE_BUFFER = 2 };

typedef struct pn_sampler_args {
  float* x;                 /* [n] latent, updated in place */
  const float* net2;        /* [2n] network output [uncond ; cond] (NULL for PN_SAMPLER_INPUT) */
  float* x_in_next;         /* [2n] or NULL */
  float* x_eval;            /* [n] Heun predictor / DPM++ 2S midpoint point */
  float* d;                 /* [n] Heun d, or [lms_ring, n] LMS derivatives */
  float* old_denoised;      /* [n] DPM++ 2M */
  const float* noise;       /* [n] caller-supplied N(0,1) draws (PN_NOISE_BUFFER) */
  int64_t n;
  uint64_t seed, draw;      /* PN_NOISE_PHILOX */
  float sigma, sigma_q, dt;
  float cfg_scale, c_in_next;
  float m1, m2, m3, m4;
  float noise_mul, noise_amp;
  float lms_coeff[4];
  int32_t mode;
  int32_t net_is_denoised;
  int32_t noise_source;
  int32_t use_old;
  int32_t lms_order, lms_ring, lms_slot;
} pn_sampler_args;

int pn_sampler_step(const pn_sampler_args* args, void* stream);
/* out[e] = N(0,1) draw number `draw` of element e under `seed`: Philox4x32-10 on the counter (e / 4, draw) with key seed,
 * Box-Muller on its two 32-bit pairs. A pure function of (seed, draw, e), independent of the launch geometry; the same
 * values pn_sampler_step adds with PN_NOISE_PHILOX. */
int pn_philox_normal(float* out, int64_t n, uint64_t seed, uint64_t draw, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PANACEA_B200_H */
