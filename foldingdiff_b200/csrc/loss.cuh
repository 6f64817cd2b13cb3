// The forward half of the training step (SURVEY.md section 8f, rank 3): forward noising, the per-feature loss terms
// and the pairwise-distance term of BertForDiffusion._get_loss_terms, evaluated on the device.
//
//   q_sample_kernel     datasets.NoisedAnglesDataset.sample_noise + __getitem__ (reference datasets.py:772-799,
//                       :801-886; host mirror foldingdiff_b200/datasets.py:113-160), elementwise, torch's op order with
//                       explicitly rounded fp32 ops so the result is bit-comparable to the host mirror
//   loss_chain_kernel   per-chain partial sums of every loss term (modelling.py:553-604, losses.py:12-62): one CTA per
//   loss_reduce_kernel  chain, fixed-order fp64 accumulation; then one fixed-order pass over the chains -> (F,) terms
//   denoise_kernel      (corrupted - s1m * eps_hat) / sa, unwrapped (modelling.py:621-628)
//   pdist_chain_kernel  CA pairwise-distance term (modelling.py:616-677, losses.py:66-150): one CTA per chain over the
//   pdist_reduce_kernel NeRF coordinates of both structures (nerf.cuh), then the mean over all pairs of the batch
//
// No float atomics anywhere: every sum has one fixed order, so two runs give the same bits.
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace fd {

constexpr int LOSS_THREADS = 256;
enum { LOSS_SMOOTH_L1 = 0, LOSS_L1 = 1 };

struct FeatureScales {
  float s[FD_MAX_FEATURES];
};

// known_noise = scale_f * z (wrapped on angular columns); corrupted = sa_b * x0 + s1m_b * known_noise (wrapped on
// angular columns).  z is the caller's draw, or element offset + (b * n_pad + n) * F + f of Philox stream `seed`.
__global__ void q_sample_kernel(const float* __restrict__ x0, long long total, int n_pad, int F,
                                const float* __restrict__ sa, const float* __restrict__ s1m, const __grid_constant__ FeatureScales scale,
                                uint32_t ang_bits, const float* __restrict__ z, uint64_t seed, uint64_t offset,
                                float* __restrict__ known, float* __restrict__ corrupted) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i % F);
    const int b = (int)(i / ((long long)n_pad * F));
    const bool ang = (ang_bits >> f) & 1u;
    const float zi = z ? z[i] : philox_normal(seed, offset + (uint64_t)i);
    float nz = __fmul_rn(zi, scale.s[f]);  // noise[..., j] *= scale (the scale rounded to fp32, like torch)
    if (ang) nz = wrap_pi(nz);
    float c = __fadd_rn(__fmul_rn(sa[b], x0[i]), __fmul_rn(s1m[b], nz));
    if (ang) c = wrap_pi(c);
    known[i] = nz;
    corrupted[i] = c;
  }
}

// torch.remainder(a, b) for float (fmod, then shift into the sign of b)
__device__ __forceinline__ float torch_rem(float a, float b) {
  float m = fmodf(a, b);
  if (m != 0.0f && ((b < 0.0f) != (m < 0.0f))) m = __fadd_rn(m, b);
  return m;
}

// One element's loss value (before the mean) for feature kind (angular?, loss); the circle term separately.
__device__ __forceinline__ float loss_elem(float pred, float tgt, bool ang, int loss) {
  if (ang && loss == LOSS_SMOOTH_L1) {  // radian_smooth_l1_loss, beta = pi / 10 (modelling.py:230-232)
    const float beta = (float)(3.14159265358979323846 / 10.0), half_beta = (float)(0.5 * 3.14159265358979323846 / 10.0);
    const float d = wrap_pi(__fsub_rn(tgt, pred));
    const float a = fabsf(d);
    return a < beta ? __fdiv_rn(__fmul_rn(0.5f, __fmul_rn(d, d)), beta) : __fsub_rn(a, half_beta);
  }
  if (ang) {  // radian_l1_loss: both reduced with %, difference folded to [-pi, pi)
    const float two_pi = 6.28318530717958647692f, pi = 3.14159265358979323846f;
    const float d = __fsub_rn(torch_rem(tgt, two_pi), torch_rem(pred, two_pi));
    return fabsf(__fsub_rn(torch_rem(__fadd_rn(d, pi), two_pi), pi));
  }
  const float a = fabsf(__fsub_rn(pred, tgt));
  if (loss == LOSS_SMOOTH_L1)  // F.smooth_l1_loss, beta = 1
    return a < 1.0f ? __fmul_rn(__fmul_rn(0.5f, a), a) : __fsub_rn(a, 0.5f);
  return a;  // F.l1_loss
}

// Block-wide fixed-order sum of one double per thread (tree over shared memory); result valid in thread 0.
__device__ __forceinline__ double block_sum_fixed(double v, double* red) {
  red[threadIdx.x] = v;
  __syncthreads();
  for (int s = LOSS_THREADS / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  const double r = red[0];
  __syncthreads();
  return r;
}

// chain b: out[b * (2F + 1) + f]      = sum over valid tokens of loss_elem(feature f)
//          out[b * (2F + 1) + F + f]  = sum over valid tokens of trunc(|pred| / pi)   (angular smooth-L1 with circle > 0)
//          out[b * (2F + 1) + 2F]     = number of valid tokens (attn_mask != 0)
__global__ void __launch_bounds__(LOSS_THREADS) loss_chain_kernel(
    const float* __restrict__ pred, const float* __restrict__ known, const float* __restrict__ mask, int n_pad, int F,
    uint32_t ang_bits, int loss, int circle, double* __restrict__ out) {
  __shared__ double red[LOSS_THREADS];
  const int b = blockIdx.x;
  const float* p = pred + (size_t)b * n_pad * F;
  const float* k = known + (size_t)b * n_pad * F;
  const float* m = mask + (size_t)b * n_pad;
  double* o = out + (size_t)b * (2 * F + 1);
  const float pi = 3.14159265358979323846f;
  for (int f = 0; f < F; ++f) {
    const bool ang = (ang_bits >> f) & 1u;
    double s = 0.0, c = 0.0;
    for (int n = threadIdx.x; n < n_pad; n += LOSS_THREADS) {
      if (m[n] == 0.0f) continue;
      const float pv = p[(size_t)n * F + f];
      s += (double)loss_elem(pv, k[(size_t)n * F + f], ang, loss);
      if (ang && circle && loss == LOSS_SMOOTH_L1) c += (double)truncf(__fdiv_rn(fabsf(pv), pi));
    }
    s = block_sum_fixed(s, red);
    c = block_sum_fixed(c, red);
    if (threadIdx.x == 0) { o[f] = s; o[F + f] = c; }
  }
  double cnt = 0.0;
  for (int n = threadIdx.x; n < n_pad; n += LOSS_THREADS) cnt += m[n] != 0.0f ? 1.0 : 0.0;
  cnt = block_sum_fixed(cnt, red);
  if (threadIdx.x == 0) o[2 * F] = cnt;
}

// terms[f] = sum_b S[b, f] / N + circle_penalty * sum_b C[b, f] / N, chains taken in order b = 0, 1, ...
__global__ void loss_reduce_kernel(const double* __restrict__ chain, int batch, int F, float circle_penalty,
                                   float* __restrict__ terms) {
  const int f = threadIdx.x;
  if (f >= F) return;
  double s = 0.0, c = 0.0, n = 0.0;
  for (int b = 0; b < batch; ++b) {
    const double* o = chain + (size_t)b * (2 * F + 1);
    s += o[f]; c += o[F + f]; n += o[2 * F];
  }
  terms[f] = (float)(s / n + (double)circle_penalty * (c / n));
}

// denoised = (corrupted - s1m_b * eps_hat) / sa_b in the reference's fp32 op order, not wrapped.
__global__ void denoise_kernel(const float* __restrict__ corrupted, const float* __restrict__ eps, long long total,
                               long long per_chain, const float* __restrict__ sa, const float* __restrict__ s1m,
                               float* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / per_chain);
    out[i] = __fdiv_rn(__fsub_rn(corrupted[i], __fmul_rn(s1m[b], eps[i])), sa[b]);
  }
}

// One CTA per chain: CA atoms (atom 3i + 1) of the denoised (a) and known (b) structures, pairs i < j < L,
// out[2b] = coef_b * sum (|a_i - a_j| - |b_i - b_j|)^2 and out[2b + 1] = L (L - 1) / 2, in fp64.
__global__ void __launch_bounds__(LOSS_THREADS) pdist_chain_kernel(
    const float* __restrict__ coords_a, const float* __restrict__ coords_b, const int* __restrict__ lengths, int n_pad,
    const float* __restrict__ coef, double* __restrict__ out) {
  __shared__ double red[LOSS_THREADS];
  __shared__ float ca[2][128][3];
  const int b = blockIdx.x;
  const int L = lengths[b];
  const float* A = coords_a + (size_t)b * n_pad * 9;
  const float* B = coords_b + (size_t)b * n_pad * 9;
  for (int i = threadIdx.x; i < L * 3; i += LOSS_THREADS) {
    const int r = i / 3, k = i % 3;
    ca[0][r][k] = A[(size_t)(3 * r + 1) * 3 + k];
    ca[1][r][k] = B[(size_t)(3 * r + 1) * 3 + k];
  }
  __syncthreads();
  double s = 0.0;
  for (int i = 0; i < L; ++i) {
    for (int j = i + 1 + threadIdx.x; j < L; j += LOSS_THREADS) {
      double da = 0.0, db = 0.0;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const double xa = (double)ca[0][i][k] - (double)ca[0][j][k], xb = (double)ca[1][i][k] - (double)ca[1][j][k];
        da += xa * xa; db += xb * xb;
      }
      const double d = sqrt(da) - sqrt(db);
      s += d * d;
    }
  }
  s = block_sum_fixed(s, red);
  if (threadIdx.x == 0) {
    out[2 * b] = (double)coef[b] * s;
    out[2 * b + 1] = 0.5 * (double)L * (double)(L - 1);
  }
}

__global__ void pdist_reduce_kernel(const double* __restrict__ chain, int batch, float* __restrict__ loss) {
  if (threadIdx.x != 0) return;
  double s = 0.0, n = 0.0;
  for (int b = 0; b < batch; ++b) { s += chain[2 * b]; n += chain[2 * b + 1]; }
  *loss = (float)(s / n);
}

}  // namespace fd
