// Fused per-evaluation update of the reference's samplers (sampling.py:96-365): denoiser scalings, classifier-free
// guidance, the sampler's update, its noise and the next network input in one elementwise pass. Every expression is
// written with explicit round-to-nearest intrinsics so that no multiply-add is contracted: the kernel rounds exactly
// where the reference's fp32 torch expressions round.
#include "common.cuh"
#include "ptx.cuh"
#include "../../include/panacea_b200.h"

namespace pn {

// ---------------------------------------------------------------- Philox4x32-10 + Box-Muller
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
    const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += W0;
    k.y += W1;
  }
  return c;
}

// N(0,1) draw `draw` of element e: counter (e / 4, draw), key seed; lanes 0/1 use the Box-Muller pair of words (x, y),
// lanes 2/3 the pair (z, w). u1 in (0, 1) (never 0), u2 in [0, 1).
__device__ __forceinline__ float philox_normal(uint64_t seed, uint64_t draw, uint64_t e) {
  const uint64_t q = e >> 2;
  const uint4 r = philox4x32_10(make_uint4((uint32_t)q, (uint32_t)(q >> 32), (uint32_t)draw, (uint32_t)(draw >> 32)),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const int lane = (int)(e & 3);
  const uint32_t a = lane < 2 ? r.x : r.z, b = lane < 2 ? r.y : r.w;
  const float u1 = __fmul_rn(__fadd_rn((float)(a >> 8), 0.5f), 5.9604644775390625e-8f);      // 2^-24
  const float u2 = __fmul_rn((float)(b >> 8), 5.9604644775390625e-8f);
  const float rad = __fsqrt_rn(__fmul_rn(-2.0f, logf(u1)));
  float s, c;
  sincospif(__fmul_rn(2.0f, u2), &s, &c);
  return __fmul_rn(rad, (lane & 1) ? s : c);
}

__global__ void philox_normal_kernel(float* __restrict__ out, size_t n, uint64_t seed, uint64_t draw) {
  pdl_prologue_done();
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x)
    out[e] = philox_normal(seed, draw, e);
}

// ---------------------------------------------------------------- the fused update
template <int MODE>
__global__ void __launch_bounds__(256) sampler_step_kernel(const pn_sampler_args a) {
  pdl_prologue_done();
  constexpr bool kStage1 = MODE == PN_SAMPLER_HEUN_A || MODE == PN_SAMPLER_DPMPP2S_A;   // x unchanged, x_eval written
  constexpr bool kAtEval = MODE == PN_SAMPLER_HEUN_B || MODE == PN_SAMPLER_DPMPP2S_B;   // network evaluated at x_eval
  const size_t n = (size_t)a.n;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const float x = a.x[e];
    float den = 0.f;
    if constexpr (MODE != PN_SAMPLER_INPUT) {
      const float xe = kAtEval ? a.x_eval[e] : x;
      float du = a.net2[e], dc = a.net2[n + e];
      if (!a.net_is_denoised) {
        // denoiser.py:28 with EpsScaling (denoiser_scaling.py:16-22): net * c_out + input * c_skip, c_out = -sigma_q
        du = __fadd_rn(__fmul_rn(du, -a.sigma_q), xe);
        dc = __fadd_rn(__fmul_rn(dc, -a.sigma_q), xe);
      }
      den = __fadd_rn(du, __fmul_rn(a.cfg_scale, __fsub_rn(dc, du)));     // sampling_utils.py:7-9
    }
    float xn = x, next_in = 0.f;
    if constexpr (MODE == PN_SAMPLER_EULER) {
      // sampling.py:103-106 (to_d, sampling_utils.py:39-40; euler_step :81-82); ancestral_euler_step :144-148
      const float d = __fdiv_rn(__fsub_rn(x, den), a.sigma);
      xn = __fadd_rn(x, __fmul_rn(a.dt, d));
    } else if constexpr (MODE == PN_SAMPLER_HEUN_A) {
      // sampling.py:103-106: the Euler predictor; HeunEDMSampler keeps d and evaluates at the predictor (:229)
      const float d = __fdiv_rn(__fsub_rn(x, den), a.sigma);
      a.d[e] = d;
      next_in = __fadd_rn(x, __fmul_rn(a.dt, d));
      a.x_eval[e] = next_in;
    } else if constexpr (MODE == PN_SAMPLER_HEUN_B) {
      // sampling.py:229-235: d_new = to_d(euler_step, next_sigma, denoised); x + (d + d_new) / 2 * dt
      const float dn = __fdiv_rn(__fsub_rn(a.x_eval[e], den), a.sigma);
      const float dp = __fdiv_rn(__fadd_rn(a.d[e], dn), 2.0f);
      xn = __fadd_rn(x, __fmul_rn(dp, a.dt));
    } else if constexpr (MODE == PN_SAMPLER_DPMPP2S_A) {
      // sampling.py:279: x2 = mult[0] * x - mult[1] * denoised
      next_in = __fsub_rn(__fmul_rn(a.m1, x), __fmul_rn(a.m2, den));
      a.x_eval[e] = next_in;
    } else if constexpr (MODE == PN_SAMPLER_DPMPP2S_B) {
      // sampling.py:281: x_dpmpp2s = mult[2] * x - mult[3] * denoised2
      xn = __fsub_rn(__fmul_rn(a.m3, x), __fmul_rn(a.m4, den));
    } else if constexpr (MODE == PN_SAMPLER_DPMPP2M) {
      // sampling.py:332-343: x_standard, or x_advanced with denoised_d = mult[2] * denoised - mult[3] * old_denoised
      const float dd = a.use_old ? __fsub_rn(__fmul_rn(a.m3, den), __fmul_rn(a.m4, a.old_denoised[e])) : den;
      xn = __fsub_rn(__fmul_rn(a.m1, x), __fmul_rn(a.m2, dd));
      a.old_denoised[e] = den;
    } else if constexpr (MODE == PN_SAMPLER_LMS) {
      // sampling.py:200-209: ds ring, x + sum(coeff * d for coeff, d in zip(coeffs, reversed(ds)))
      const float d = __fdiv_rn(__fsub_rn(x, den), a.sigma);
      a.d[(size_t)a.lms_slot * n + e] = d;
      float acc = __fmul_rn(a.lms_coeff[0], d);
      for (int j = 1; j < a.lms_order; ++j) {
        const int s = (a.lms_slot - j + a.lms_ring) % a.lms_ring;
        acc = __fadd_rn(acc, __fmul_rn(a.lms_coeff[j], a.d[(size_t)s * n + e]));
      }
      xn = __fadd_rn(x, acc);
    }
    if constexpr (!kStage1) {
      // sampling.py:99-100 (EDM churn of the step that follows) and :151-155 (ancestral noise):
      // x + (z * s_noise) * amplitude
      if (a.noise_source != PN_NOISE_NONE) {
        const float z = a.noise_source == PN_NOISE_BUFFER ? a.noise[e] : philox_normal(a.seed, a.draw, e);
        xn = __fadd_rn(xn, __fmul_rn(__fmul_rn(z, a.noise_mul), a.noise_amp));
      }
      a.x[e] = xn;
      next_in = xn;
    }
    if (a.x_in_next) {
      const float v = __fmul_rn(next_in, a.c_in_next);      // denoiser.py:28 input * c_in, CFG batch doubling
      a.x_in_next[e] = v;
      a.x_in_next[n + e] = v;
    }
  }
}

static inline int sampler_grid(size_t total) {
  size_t g = (total + 255) / 256;
  const size_t cap = (size_t)16 * sm_count();
  if (g > cap) g = cap;
  return (int)(g < 1 ? 1 : g);
}

}  // namespace pn

using namespace pn;

extern "C" int pn_sampler_step(const pn_sampler_args* args, void* stream_v) {
  PN_REQUIRE(args && args->x && args->n > 0, "pn_sampler_step: bad arguments");
  const pn_sampler_args& a = *args;
  const int m = a.mode;
  PN_REQUIRE(m >= PN_SAMPLER_INPUT && m <= PN_SAMPLER_LMS, "pn_sampler_step: mode %d", m);
  PN_REQUIRE(m == PN_SAMPLER_INPUT || a.net2, "pn_sampler_step: net2 is required");
  PN_REQUIRE(!(m == PN_SAMPLER_EULER || m == PN_SAMPLER_HEUN_A || m == PN_SAMPLER_HEUN_B || m == PN_SAMPLER_LMS) || a.sigma > 0.f,
             "pn_sampler_step: sigma must be positive");
  PN_REQUIRE(!(m == PN_SAMPLER_HEUN_A || m == PN_SAMPLER_HEUN_B || m == PN_SAMPLER_DPMPP2S_A || m == PN_SAMPLER_DPMPP2S_B) || a.x_eval,
             "pn_sampler_step: x_eval is required");
  PN_REQUIRE(!(m == PN_SAMPLER_HEUN_A || m == PN_SAMPLER_HEUN_B || m == PN_SAMPLER_LMS) || a.d, "pn_sampler_step: d is required");
  PN_REQUIRE(m != PN_SAMPLER_DPMPP2M || a.old_denoised, "pn_sampler_step: old_denoised is required");
  PN_REQUIRE(m != PN_SAMPLER_LMS || (a.lms_ring >= 1 && a.lms_ring <= 4 && a.lms_order >= 1 && a.lms_order <= a.lms_ring &&
                                     a.lms_slot >= 0 && a.lms_slot < a.lms_ring),
             "pn_sampler_step: LMS order %d / ring %d / slot %d", a.lms_order, a.lms_ring, a.lms_slot);
  PN_REQUIRE(a.noise_source >= PN_NOISE_NONE && a.noise_source <= PN_NOISE_BUFFER, "pn_sampler_step: noise_source %d", a.noise_source);
  PN_REQUIRE(a.noise_source != PN_NOISE_BUFFER || a.noise, "pn_sampler_step: noise buffer is required");
  const dim3 grid(sampler_grid((size_t)a.n)), block(256);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream_v);
  cudaError_t err = cudaSuccess;
  switch (m) {
    case PN_SAMPLER_INPUT: err = launch_kernel(sampler_step_kernel<PN_SAMPLER_INPUT>, grid, block, 0, st, 1, a); break;
    case PN_SAMPLER_EULER: err = launch_kernel(sampler_step_kernel<PN_SAMPLER_EULER>, grid, block, 0, st, 1, a); break;
    case PN_SAMPLER_HEUN_A: err = launch_kernel(sampler_step_kernel<PN_SAMPLER_HEUN_A>, grid, block, 0, st, 1, a); break;
    case PN_SAMPLER_HEUN_B: err = launch_kernel(sampler_step_kernel<PN_SAMPLER_HEUN_B>, grid, block, 0, st, 1, a); break;
    case PN_SAMPLER_DPMPP2S_A: err = launch_kernel(sampler_step_kernel<PN_SAMPLER_DPMPP2S_A>, grid, block, 0, st, 1, a); break;
    case PN_SAMPLER_DPMPP2S_B: err = launch_kernel(sampler_step_kernel<PN_SAMPLER_DPMPP2S_B>, grid, block, 0, st, 1, a); break;
    case PN_SAMPLER_DPMPP2M: err = launch_kernel(sampler_step_kernel<PN_SAMPLER_DPMPP2M>, grid, block, 0, st, 1, a); break;
    default: err = launch_kernel(sampler_step_kernel<PN_SAMPLER_LMS>, grid, block, 0, st, 1, a); break;
  }
  PN_CHECK_CUDA(err);
  PN_CHECK_CUDA(cudaGetLastError());
  return PN_OK;
}

extern "C" int pn_philox_normal(float* out, int64_t n, uint64_t seed, uint64_t draw, void* stream_v) {
  PN_REQUIRE(out && n > 0, "pn_philox_normal: bad arguments");
  PN_CHECK_CUDA(launch_kernel(philox_normal_kernel, dim3(sampler_grid((size_t)n)), dim3(256), 0,
                              reinterpret_cast<cudaStream_t>(stream_v), 1, out, (size_t)n, seed, draw));
  return PN_OK;
}
