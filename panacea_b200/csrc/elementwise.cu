// Small HBM-bound helpers of the denoising path: layout changes at the NCHW module boundary, nearest 2x
// upsampling, skip concatenation, timestep embedding, the tiny time-embedding linears, stride-2 im2col and the
// fused classifier-free-guidance + Euler update of the sampler.
#include "common.cuh"
#include "ptx.cuh"
#include "operand.cuh"
#include "../../include/panacea_b200.h"

namespace pn {

// ---------------------------------------------------------------- [F, A, B] -> out[f, b, off + a] (row stride ld)
__global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int A, int B, long long in_ld,
                                 long long ld, int off) {
  pdl_prologue_done();
  __shared__ float tile[32][33];
  const int f = blockIdx.z;
  const int b0 = blockIdx.x * 32, a0 = blockIdx.y * 32;
  const float* src = in + (size_t)f * A * in_ld;
  float* dst = out + (size_t)f * B * ld;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int a = a0 + i, b = b0 + threadIdx.x;
    if (a < A && b < B) tile[i][threadIdx.x] = src[(size_t)a * in_ld + b];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int b = b0 + i, a = a0 + threadIdx.x;
    if (a < A && b < B) dst[(size_t)b * ld + off + a] = tile[threadIdx.x][i];
  }
}

// ---------------------------------------------------------------- nearest 2x upsample, fp32 -> GEMM operand
template <int OP>
__global__ void upsample2x_kernel(const float* __restrict__ x, void* __restrict__ y, int F, int H, int W, int C) {
  pdl_prologue_done();
  const int c8n = C / 8;
  const size_t total = (size_t)F * (2 * H) * (2 * W) * c8n;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const int c8 = (int)(e % c8n);
    size_t r = e / c8n;
    const int ox = (int)(r % (2 * W)); r /= (2 * W);
    const int oy = (int)(r % (2 * H));
    const int f = (int)(r / (2 * H));
    const float* src = x + (((size_t)f * H + (oy >> 1)) * W + (ox >> 1)) * C + c8 * 8;
    const float4 a = *reinterpret_cast<const float4*>(src);
    const float4 b = *reinterpret_cast<const float4*>(src + 4);
    const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    store_op8<OP>(y, ((size_t)f * 2 * H + oy) * 2 * W + ox, C, c8 * 8, v);
  }
}

// ---------------------------------------------------------------- out = cat(h, skip (+ ctrl)) along channels
__global__ void concat_add_kernel(const float* __restrict__ h, const float* __restrict__ skip,
                                  const float* __restrict__ ctrl, float* __restrict__ out, long long rows, int C1,
                                  int C2) {
  pdl_prologue_done();
  const int Ct = C1 + C2;
  const int c4n = Ct / 4;
  const size_t total = (size_t)rows * c4n;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % c4n) * 4;
    const size_t r = e / c4n;
    float4 v;
    if (c < C1) {
      v = *reinterpret_cast<const float4*>(h + r * C1 + c);
    } else {
      v = *reinterpret_cast<const float4*>(skip + r * C2 + (c - C1));
      if (ctrl) {
        const float4 k = *reinterpret_cast<const float4*>(ctrl + r * C2 + (c - C1));
        v.x += k.x; v.y += k.y; v.z += k.z; v.w += k.w;
      }
    }
    *reinterpret_cast<float4*>(out + r * Ct + c) = v;
  }
}

__global__ void add_inplace_kernel(float* __restrict__ x, const float* __restrict__ y, size_t n4) {
  pdl_prologue_done();
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n4; e += (size_t)gridDim.x * blockDim.x) {
    float4 a = reinterpret_cast<float4*>(x)[e];
    const float4 b = reinterpret_cast<const float4*>(y)[e];
    a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    reinterpret_cast<float4*>(x)[e] = a;
  }
}

// fp32 [rows, C] -> GEMM operand [rows, C] (bf16) or [rows, 3C] (split3)
template <int OP>
__global__ void cast_operand_kernel(const float* __restrict__ x, void* __restrict__ y, size_t rows, int C) {
  pdl_prologue_done();
  const int c4n = C / 4;
  const size_t n4 = rows * (size_t)c4n;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n4; e += (size_t)gridDim.x * blockDim.x) {
    const float4 a = reinterpret_cast<const float4*>(x)[e];
    const float v[4] = {a.x, a.y, a.z, a.w};
    store_op4<OP>(y, e / c4n, C, (int)(e % c4n) * 4, v);
  }
}

// GEGLU on an fp32 GEMM output whose columns are packed in blocks of 32 (16 value columns, then the 16 gate columns
// of the same outputs — the layout of pn_gemm's fused GEGLU epilogue): out[row, 16 b + i] = in[row, 32 b + i] *
// gelu_erf(in[row, 32 b + 16 + i]) with the exact erf GELU of the reference (attention.py:97-99). Parity mode only.
template <int OP>
__global__ void geglu_operand_kernel(const float* __restrict__ in, void* __restrict__ y, size_t rows, int inner) {
  pdl_prologue_done();
  const int c4n = inner / 4;
  const size_t n4 = rows * (size_t)c4n;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n4; e += (size_t)gridDim.x * blockDim.x) {
    const size_t row = e / c4n;
    const int col = (int)(e % c4n) * 4;
    const float* src = in + row * (size_t)(2 * inner) + (col / 16) * 32 + (col % 16);
    const float4 val = *reinterpret_cast<const float4*>(src);
    const float4 gate = *reinterpret_cast<const float4*>(src + 16);
    const float vv[4] = {val.x, val.y, val.z, val.w}, gg[4] = {gate.x, gate.y, gate.z, gate.w};
    float o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = vv[i] * (0.5f * gg[i] * (1.0f + erff(gg[i] * 0.70710678118654752f)));
    store_op4<OP>(y, row, inner, col, o);
  }
}

// ---------------------------------------------------------------- sinusoidal timestep embedding
// util.py:224-248: emb[n] = [cos(t f_k), sin(t f_k)], f_k = exp(-ln(10000) k / half)
// freqs (optional): the caller's fp32 table of the dim/2 frequencies (the host computes it with the reference's own
// expression, so the arguments t * f_k are bit-identical to the reference's — t is up to 999, an ulp of f_k matters).
__global__ void timestep_embedding_kernel(const long long* __restrict__ t, float* __restrict__ out, int n, int dim,
                                          const float* __restrict__ freqs) {
  pdl_prologue_done();
  const int half = dim / 2;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * half) return;
  const int row = i / half, k = i - row * half;
  const float freq = freqs ? freqs[k] : expf(-9.210340371976184f * (float)k / (float)half);
  const float arg = (float)t[row] * freq;
  out[(size_t)row * dim + k] = cosf(arg);
  out[(size_t)row * dim + half + k] = sinf(arg);
  if ((dim & 1) && k == 0) out[(size_t)row * dim + dim - 1] = 0.f;
}

// ---------------------------------------------------------------- small-M linear (time-embedding MLPs)
// y[m, n] = act_out( b[n] + sum_k W[n,k] * act_in(x[m,k]) ), fp32 activations, bf16 weights, M <= 32.
// One warp computes 4 output columns for all rows (weights are the traffic; x stays in L1/L2).
template <typename TW>
__device__ __forceinline__ float2 load_w2(const TW* p);
template <>
__device__ __forceinline__ float2 load_w2<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p));
}
template <>
__device__ __forceinline__ float2 load_w2<float>(const float* p) { return *reinterpret_cast<const float2*>(p); }

template <int MAXM, typename TW>
__global__ void __launch_bounds__(128) linear_small_kernel(const float* __restrict__ x, const TW* __restrict__ W,
                                                           const float* __restrict__ bias, float* __restrict__ y, int M,
                                                           int N, int K, long long ldy, int silu_in, int silu_out) {
  pdl_prologue_done();
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int n0 = warp * 4;
  if (n0 >= N) return;
  float acc[MAXM][4];
#pragma unroll
  for (int m = 0; m < MAXM; ++m)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[m][j] = 0.f;
  for (int k = lane * 2; k < K; k += 64) {
    // all loads of the iteration first (4 weight rows, MAXM activation rows), then the math: issued one row at a time
    // behind its FMAs the MAXM activation loads were MAXM serial L2 round trips per iteration (178 us for the
    // 1280 x 1280 time-embedding Linear on 16 rows)
    constexpr int MB = MAXM < 16 ? MAXM : 16;          // activation rows loaded per batch
    float2 w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = min(n0 + j, N - 1);
      w[j] = load_w2<TW>(W + (size_t)n * K + k);
    }
#pragma unroll
    for (int m0 = 0; m0 < MAXM; m0 += MB) {
      float2 xv[MB];
#pragma unroll
      for (int m = 0; m < MB; ++m) xv[m] = *reinterpret_cast<const float2*>(x + (size_t)(m0 + m < M ? m0 + m : 0) * K + k);
#pragma unroll
      for (int m = 0; m < MB; ++m) {
        float2 v = xv[m];
        if (silu_in) { v.x = silu(v.x); v.y = silu(v.y); }
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[m0 + m][j] += v.x * w[j].x + v.y * w[j].y;
      }
    }
  }
#pragma unroll
  for (int m = 0; m < MAXM; ++m)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc[m][j] += __shfl_xor_sync(0xffffffffu, acc[m][j], o);
  if (lane == 0) {
    for (int m = 0; m < M && m < MAXM; ++m)
      for (int j = 0; j < 4; ++j)
        if (n0 + j < N) {
          float v = acc[m][j] + (bias ? bias[n0 + j] : 0.f);
          y[(size_t)m * ldy + n0 + j] = silu_out ? silu(v) : v;
        }
  }
}

// ---------------------------------------------------------------- stride-2 3x3 im2col, fp32 NHWC -> operand [rows*9, C]
// (viewed by the GEMM as [rows, 9*C] or [rows, 9*3C]: every tap is one operand row)
template <int OP>
__global__ void im2col_s2_kernel(const float* __restrict__ x, void* __restrict__ out, int F, int H, int W, int C,
                                 int Ho, int Wo, int pad) {
  pdl_prologue_done();
  const int c8n = C / 8;
  const size_t total = (size_t)F * Ho * Wo * 9 * c8n;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const int c8 = (int)(e % c8n);
    size_t r = e / c8n;
    const int tap = (int)(r % 9); r /= 9;
    const int ox = (int)(r % Wo); r /= Wo;
    const int oy = (int)(r % Ho);
    const int f = (int)(r / Ho);
    const int iy = oy * 2 - pad + tap / 3, ix = ox * 2 - pad + tap % 3;
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
      const float* src = x + (((size_t)f * H + iy) * W + ix) * C + c8 * 8;
      const float4 a = *reinterpret_cast<const float4*>(src);
      const float4 b = *reinterpret_cast<const float4*>(src + 4);
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
    store_op8<OP>(out, (((size_t)f * Ho + oy) * Wo + ox) * 9 + tap, C, c8 * 8, v);
  }
}

// ---------------------------------------------------------------- scaled copies (sampler input, CFG batch doubling)
__global__ void scale_dup_kernel(const float* __restrict__ x, float* __restrict__ out, size_t n, float s, int copies) {
  pdl_prologue_done();
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const float v = x[e] * s;
    for (int c = 0; c < copies; ++c) out[(size_t)c * n + e] = v;
  }
}

// ---------------------------------------------------------------- row softmax, fp32 scores -> bf16 probabilities
// The single-head, C-wide attention of the VAE mid block (reference model.py:374-414: SDPA over all h*w tokens with
// head_dim = C = 512) is run as GEMMs (S = q k^T, O = P v) around this kernel: out[r, :] = softmax(scale * in[r, :]).
// One CTA per row; the row's exponentials are kept in shared memory between the sum and the normalised store.
__global__ void __launch_bounds__(256) softmax_rows_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, int N,
                                                           long long ld_in, long long ld_out, float scale_log2) {
  pdl_prologue_done();
  extern __shared__ float sm_row[];
  __shared__ float red[8];
  const float* src = in + (long long)blockIdx.x * ld_in;
  __nv_bfloat16* dst = out + (long long)blockIdx.x * ld_out;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float m = -INFINITY;
  for (int i = threadIdx.x * 4; i < N; i += 1024) {
    const float4 v = *reinterpret_cast<const float4*>(src + i);
    *reinterpret_cast<float4*>(sm_row + i) = v;
    m = fmaxf(fmaxf(m, fmaxf(v.x, v.y)), fmaxf(v.z, v.w));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) red[warp] = m;
  __syncthreads();
  m = red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
  __syncthreads();
  const float nm = -m * scale_log2;
  float s = 0.f;
  for (int i = threadIdx.x * 4; i < N; i += 1024) {
    float4 v = *reinterpret_cast<float4*>(sm_row + i);
    v.x = exp2f(fmaf(v.x, scale_log2, nm)); v.y = exp2f(fmaf(v.y, scale_log2, nm));
    v.z = exp2f(fmaf(v.z, scale_log2, nm)); v.w = exp2f(fmaf(v.w, scale_log2, nm));
    *reinterpret_cast<float4*>(sm_row + i) = v;
    s += (v.x + v.y) + (v.z + v.w);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) red[warp] = s;
  __syncthreads();
  s = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) s += red[w];
  const float inv = 1.f / s;
  for (int i = threadIdx.x * 4; i < N; i += 1024) {
    const float4 v = *reinterpret_cast<float4*>(sm_row + i);
    *reinterpret_cast<uint2*>(dst + i) = make_uint2(pack_bf16x2(v.x * inv, v.y * inv), pack_bf16x2(v.z * inv, v.w * inv));
  }
}

// ---------------------------------------------------------------- content fingerprint of a device buffer
// Two order-independent 64-bit sums over the 32-bit words (plain sum, position-weighted sum). The conditioning cache of
// the wrapper keys on CONTENT with it: tensor addresses are recycled by the allocator and the reference's guider
// rebuilds its torch.cat-ed dict every step, so neither identity nor address says whether the BEV hint / text changed.
__global__ void fingerprint_kernel(const uint32_t* __restrict__ x, size_t nwords, unsigned long long* __restrict__ out2) {
  pdl_prologue_done();
  unsigned long long s1 = 0ull, s2 = 0ull;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nwords; i += (size_t)gridDim.x * blockDim.x) {
    const unsigned long long w = x[i];
    s1 += w;
    s2 += w * ((unsigned long long)i * 0x9E3779B97F4A7C15ull + 0xD1B54A32D192ED03ull);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&out2[0], s1);
    atomicAdd(&out2[1], s2);
  }
}

static inline int grid_for(size_t total, int threads = 256) {
  size_t g = (total + threads - 1) / threads;
  const size_t cap = (size_t)16 * sm_count();
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace pn

using namespace pn;

extern "C" int pn_transpose_f32(const float* in, float* out, int64_t batch, int64_t A, int64_t B, int64_t in_ld, int64_t out_ld,
                                int64_t out_off, void* stream_v) {
  PN_REQUIRE(in && out && batch > 0 && A > 0 && B > 0 && in_ld >= B && out_ld >= out_off + A, "pn_transpose_f32: bad arguments");
  PN_REQUIRE(batch <= 65535, "pn_transpose_f32: batch too large");
  dim3 grid((unsigned)((B + 31) / 32), (unsigned)((A + 31) / 32), (unsigned)batch);
  launch_kernel(transpose_kernel, dim3(grid), dim3(dim3(32, 8)), 0, reinterpret_cast<cudaStream_t>(stream_v), 1, in, out, (int)A, (int)B, (long long)in_ld,
                                                                                         (long long)out_ld, (int)out_off);
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}

extern "C" int pn_upsample2x(const float* x, void* y, int64_t frames, int64_t H, int64_t W, int64_t C, int operand_mode,
                             void* stream_v) {
  PN_REQUIRE(x && y && frames > 0 && H > 0 && W > 0 && C > 0 && C % 8 == 0, "pn_upsample2x: bad arguments");
  PN_REQUIRE(operand_mode >= 0 && operand_mode <= 2, "pn_upsample2x: operand_mode %d", operand_mode);
  const size_t total = (size_t)frames * 4 * H * W * (C / 8);
  PN_DISPATCH_OP(operand_mode, (launch_kernel(upsample2x_kernel<OP>, dim3(grid_for(total)), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream_v), 1, 
      x, y, (int)frames, (int)H, (int)W, (int)C)));
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}

extern "C" int pn_concat_add(const float* h, const float* skip, const float* ctrl, float* out, int64_t rows, int64_t C1,
                             int64_t C2, void* stream_v) {
  PN_REQUIRE(h && skip && out && rows > 0 && C1 % 4 == 0 && C2 % 4 == 0 && C1 > 0 && C2 > 0, "pn_concat_add: bad arguments");
  const size_t total = (size_t)rows * ((C1 + C2) / 4);
  launch_kernel(concat_add_kernel, dim3(grid_for(total)), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream_v), 1, h, skip, ctrl, out, rows,
                                                                                           (int)C1, (int)C2);
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}

extern "C" int pn_add_inplace(float* x, const float* y, int64_t n, void* stream_v) {
  PN_REQUIRE(x && y && n > 0 && n % 4 == 0, "pn_add_inplace: bad arguments");
  launch_kernel(add_inplace_kernel, dim3(grid_for((size_t)n / 4)), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream_v), 1, x, y, (size_t)n / 4);
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}

extern "C" int pn_cast_operand(const float* x, void* y, int64_t rows, int64_t C, int operand_mode, void* stream_v) {
  PN_REQUIRE(x && y && rows > 0 && C > 0 && C % 4 == 0, "pn_cast_operand: bad arguments");
  PN_REQUIRE(operand_mode == PN_OP_BF16 || operand_mode == PN_OP_SPLIT3, "pn_cast_operand: operand_mode %d", operand_mode);
  const size_t n4 = (size_t)rows * (size_t)(C / 4);
  PN_DISPATCH_OP(operand_mode, (launch_kernel(cast_operand_kernel<OP>, dim3(grid_for(n4)), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream_v), 1, 
      x, y, (size_t)rows, (int)C)));
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}

extern "C" int pn_geglu_operand(const float* in, void* y, int64_t rows, int64_t inner, int operand_mode, void* stream_v) {
  PN_REQUIRE(in && y && rows > 0 && inner > 0 && inner % 16 == 0, "pn_geglu_operand: bad arguments");
  PN_REQUIRE(operand_mode >= 0 && operand_mode <= 2, "pn_geglu_operand: operand_mode %d", operand_mode);
  const size_t n4 = (size_t)rows * (size_t)(inner / 4);
  PN_DISPATCH_OP(operand_mode, (launch_kernel(geglu_operand_kernel<OP>, dim3(grid_for(n4)), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream_v), 1, 
      in, y, (size_t)rows, (int)inner)));
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}

extern "C" int pn_timestep_embedding(const int64_t* t, float* out, int64_t n, int64_t dim, const float* freqs,
                                     void* stream_v) {
  PN_REQUIRE(t && out && n > 0 && dim >= 2, "pn_timestep_embedding: bad arguments");
  const int total = (int)(n * (dim / 2));
  launch_kernel(timestep_embedding_kernel, dim3((total + 255) / 256), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream_v), 1, 
      reinterpret_cast<const long long*>(t), out, (int)n, (int)dim, freqs);
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}

extern "C" int pn_linear_small(const float* x, const void* W_any, int w_is_f32, const float* bias, float* y, int64_t M,
                               int64_t N, int64_t K, int64_t ldy, int silu_in, int silu_out, void* stream_v) {
  PN_REQUIRE(x && W_any && y, "pn_linear_small: null pointer");
  PN_REQUIRE(M > 0 && M <= 32 && N > 0 && K > 0 && K % 2 == 0 && ldy >= N, "pn_linear_small: M=%lld N=%lld K=%lld unsupported",
             (long long)M, (long long)N, (long long)K);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream_v);
  const int warps = (int)((N + 3) / 4);
  const int blocks = (warps * 32 + 127) / 128;
#define PN_LS(TW)                                                                                                               \
  do {                                                                                                                          \
    const TW* W = reinterpret_cast<const TW*>(W_any);                                                                          \
    if (M <= 8) launch_kernel(linear_small_kernel<8, TW>, dim3(blocks), dim3(128), 0, st, 1, x, W, bias, y, (int)M, (int)N, (int)K, ldy, silu_in, silu_out);        \
    else if (M <= 16) launch_kernel(linear_small_kernel<16, TW>, dim3(blocks), dim3(128), 0, st, 1, x, W, bias, y, (int)M, (int)N, (int)K, ldy, silu_in, silu_out); \
    else launch_kernel(linear_small_kernel<32, TW>, dim3(blocks), dim3(128), 0, st, 1, x, W, bias, y, (int)M, (int)N, (int)K, ldy, silu_in, silu_out);              \
  } while (0)
  if (w_is_f32) PN_LS(float);
  else PN_LS(__nv_bfloat16);
#undef PN_LS
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}

extern "C" int pn_im2col3x3_s2(const float* x, void* out, int64_t frames, int64_t H, int64_t W, int64_t C, int pad,
                               int operand_mode, void* stream_v) {
  PN_REQUIRE(x && out && frames > 0 && H > 0 && W > 0 && C > 0 && C % 8 == 0, "pn_im2col3x3_s2: bad arguments");
  PN_REQUIRE(operand_mode == PN_OP_BF16 || operand_mode == PN_OP_SPLIT3, "pn_im2col3x3_s2: operand_mode %d", operand_mode);
  PN_REQUIRE(pad == 0 || pad == 1, "pn_im2col3x3_s2: pad must be 1 (symmetric) or 0 (zero row/column appended at the far edges)");
  // pad 1: Conv2d(k3, s2, padding=1); pad 0: F.pad(x, (0,1,0,1)) + Conv2d(k3, s2, padding=0) (the VAE encoder's Downsample)
  const int Ho = (int)((H + 2 * pad + (1 - pad) - 3) / 2 + 1), Wo = (int)((W + 2 * pad + (1 - pad) - 3) / 2 + 1);
  const size_t total = (size_t)frames * Ho * Wo * 9 * (C / 8);
  PN_DISPATCH_OP(operand_mode, (launch_kernel(im2col_s2_kernel<OP>, dim3(grid_for(total)), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream_v), 1, 
      x, out, (int)frames, (int)H, (int)W, (int)C, Ho, Wo, pad)));
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}

extern "C" int pn_scale_dup(const float* x, float* out, int64_t n, float s, int copies, void* stream_v) {
  PN_REQUIRE(x && out && n > 0 && copies >= 1, "pn_scale_dup: bad arguments");
  launch_kernel(scale_dup_kernel, dim3(grid_for((size_t)n)), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream_v), 1, x, out, (size_t)n, s, copies);
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}

extern "C" int pn_fingerprint(const void* x, int64_t nbytes, uint64_t* out2, void* stream_v) {
  PN_REQUIRE(x && out2 && nbytes > 0 && nbytes % 4 == 0, "pn_fingerprint: bad arguments");
  PN_REQUIRE((reinterpret_cast<uintptr_t>(x) & 3) == 0, "pn_fingerprint: pointer must be 4-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream_v);
  PN_CHECK_CUDA(cudaMemsetAsync(out2, 0, 16, st));
  const size_t nwords = (size_t)nbytes / 4;
  launch_kernel(fingerprint_kernel, dim3(grid_for(nwords)), dim3(256), 0, st, 1, reinterpret_cast<const uint32_t*>(x), nwords,
                                                      reinterpret_cast<unsigned long long*>(out2));
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}

extern "C" int pn_softmax_rows(const float* in, void* out_bf16, int64_t rows, int64_t N, int64_t ld_in, int64_t ld_out, float scale,
                               void* stream_v) {
  PN_REQUIRE(in && out_bf16 && rows > 0 && N > 0 && N % 4 == 0 && ld_in >= N && ld_out >= N && ld_in % 4 == 0 && ld_out % 4 == 0,
             "pn_softmax_rows: bad arguments");
  PN_REQUIRE(N * 4 <= 200 * 1024, "pn_softmax_rows: N=%lld exceeds the shared-memory row buffer", (long long)N);
  PN_REQUIRE(rows < (1ll << 31), "pn_softmax_rows: too many rows");
  const size_t smem = (size_t)N * sizeof(float);
  const int rc = ensure_dyn_smem(reinterpret_cast<const void*>(&softmax_rows_kernel), smem);
  if (rc != PN_OK) return rc;
  launch_kernel(softmax_rows_kernel, dim3((unsigned)rows), dim3(256), smem, reinterpret_cast<cudaStream_t>(stream_v), 1, 
      in, reinterpret_cast<__nv_bfloat16*>(out_bf16), (int)N, ld_in, ld_out, scale * 1.4426950408889634f);
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}
