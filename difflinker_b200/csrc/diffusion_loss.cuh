// Diffusion objective, evaluation half (EDM.forward, reference src/edm.py:41-124): the q(z_t | x, h) sample that feeds one
// Dynamics.forward, and the per-molecule sums of the loss that follow it. The per-molecule scalars (alpha_t, sigma_t,
// alpha_T, ...) come from the caller, computed with the reference's own torch ops; the final combinations of the sums
// (l2, loss_term_t, loss_term_0, batch means) are per-molecule scalar arithmetic the caller does as well.
#pragma once
#include "kernels_simt.cuh"

namespace dl {

// z_t = xh*fragment_mask + (alpha_t*xh + sigma_t*eps_t)*linker_mask with eps_t = noise*linker_mask (edm.py:64-75,
// utils.py:189-192); eps_t is stored beside z_t for the loss kernel. One thread per element. The products and sums are
// rounded one at a time (no FMA contraction), as torch evaluates them, so z_t is the reference's to the bit.
// coef is (DL_LOSS_COEFS, B): row k holds coefficient k of every molecule.
__global__ void k_qsample(int n_total, int N, int xd, const float* __restrict__ xh, const float* __restrict__ fm,
                          const float* __restrict__ lm, const float* __restrict__ noise, NoiseRng rng,
                          const float* __restrict__ coef, float* __restrict__ z, float* __restrict__ eps) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_total * xd) return;
  const int g = idx / xd, d = idx - g * xd, b = g / N, B = n_total / N;
  const float l = lm[g];
  const float e = (rng.on ? noise_draw(rng, 0, g, d) : noise[idx]) * l;
  const float v = xh[idx];
  const float zt = __fadd_rn(__fmul_rn(coef[DL_LOSS_ALPHA_T * B + b], v), __fmul_rn(coef[DL_LOSS_SIGMA_T * B + b], e));
  z[idx] = __fadd_rn(__fmul_rn(v, fm[g]), __fmul_rn(zt, l));
  eps[idx] = e;
}

struct LossArgs {
  int N, F;
  const float* xh;       // (B,N,3+F) normalised x, h
  const float* z;        // (B,N,3+F) z_t
  const float* eps;      // (B,N,3+F) eps_t (masked)
  const float* out;      // (B,N,3+F) Dynamics.forward output (not yet multiplied by linker_mask)
  const float* lm;       // (B,N) linker_mask
  const float* coef;     // (DL_LOSS_COEFS, B)
  float norm1, bias1;
  float* terms;          // (B, DL_LOSS_TERMS)
};

constexpr int LOSS_THREADS = 256;
constexpr int LOSS_SUMS = 6;
constexpr int MAX_F = MAX_XHD - 3;

// One CTA per molecule. Every thread accumulates a fixed, strided subset of the molecule's elements in index order, then
// the CTA adds the per-thread partials in a fixed tree: the result does not depend on scheduling (no float atomics).
__global__ void __launch_bounds__(LOSS_THREADS) k_diffusion_loss(LossArgs a) {
  __shared__ float red[LOSS_SUMS][LOSS_THREADS];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int N = a.N, F = a.F, xd = 3 + F, B = gridDim.x;
  const float sigma_t = a.coef[DL_LOSS_SIGMA_T * B + b];
  const float alpha_T = a.coef[DL_LOSS_ALPHA_1 * B + b];
  const float sigma2_T = a.coef[DL_LOSS_SIGMA2_1 * B + b];
  const float log_inv_sigma_T = a.coef[DL_LOSS_LOG_INV_SIGMA_1 * B + b];
  const size_t base = (size_t)b * N * xd;
  float err = 0.f, err_x = 0.f, nsq = 0.f, mu_x2 = 0.f, kl_h = 0.f, log_p_h = 0.f;
  // elementwise sums: ||eps_t - eps_hat||^2 (edm.py:88), its x part (edm.py:292), ||eps_hat||^2 (edm.py:104),
  // ||alpha_T x||^2 over all rows and the Gaussian KL of the h part over all rows, padding included (edm.py:244-270, 434-448)
  for (int i = tid; i < N * xd; i += LOSS_THREADS) {
    const int n = i / xd, d = i - n * xd;
    const float l = a.lm[(size_t)b * N + n];
    const float eh = __fmul_rn(a.out[base + i], l);
    const float df = __fsub_rn(a.eps[base + i], eh);
    const float sq = __fmul_rn(df, df);
    err += sq;
    nsq += __fmul_rn(eh, eh);
    const float mu = __fmul_rn(alpha_T, a.xh[base + i]);
    const float mu2 = __fmul_rn(mu, mu);
    if (d < 3) {
      err_x += sq;
      mu_x2 += mu2;
    } else {
      // log(1/sigma_T) + 0.5*(sigma_T^2 + mu^2)/1 - 0.5, rounded step by step as torch does
      kl_h += __fsub_rn(__fadd_rn(log_inv_sigma_T, __fmul_rn(0.5f, __fadd_rn(sigma2_T, mu2))), 0.5f);
    }
  }
  // categorical term of log p(h | z_0) (edm.py:294-318), one row per thread: log of the normal mass of [0.5, 1.5] around
  // each estimated class value, normalised by a max-shifted logsumexp over the F classes, weighted by h * linker_mask
  const float sigma0 = __fmul_rn(sigma_t, a.norm1);
  for (int n = tid; n < N; n += LOSS_THREADS) {
    const float* zr = a.z + base + (size_t)n * xd + 3;
    const float* hr = a.xh + base + (size_t)n * xd + 3;
    const float l = a.lm[(size_t)b * N + n];
    float lp[MAX_F];                                         // fully unrolled below: stays in registers
    float m = -INFINITY;
#pragma unroll
    for (int f = 0; f < MAX_F; ++f) {
      if (f >= F) break;
      const float c = __fsub_rn(__fadd_rn(__fmul_rn(zr[f], a.norm1), a.bias1), 1.f);
      const float hi = 0.5f * (1.f + erff(__fdiv_rn(__fdiv_rn(__fadd_rn(c, 0.5f), sigma0), 1.41421356237309515f)));
      const float lo = 0.5f * (1.f + erff(__fdiv_rn(__fdiv_rn(__fsub_rn(c, 0.5f), sigma0), 1.41421356237309515f)));
      lp[f] = logf(__fadd_rn(__fsub_rn(hi, lo), 1e-10f));
      m = fmaxf(m, lp[f]);
    }
    float s = 0.f;
#pragma unroll
    for (int f = 0; f < MAX_F; ++f)
      if (f < F) s += expf(lp[f] - m);
    const float log_z = m + logf(s);
#pragma unroll
    for (int f = 0; f < MAX_F; ++f) {
      if (f >= F) break;
      const float h = __fadd_rn(__fmul_rn(hr[f], a.norm1), a.bias1);
      log_p_h += __fmul_rn(__fmul_rn(__fsub_rn(lp[f], log_z), h), l);
    }
  }
  red[0][tid] = err; red[1][tid] = err_x; red[2][tid] = nsq; red[3][tid] = mu_x2; red[4][tid] = kl_h; red[5][tid] = log_p_h;
  __syncthreads();
  for (int w = LOSS_THREADS / 2; w > 0; w >>= 1) {
    if (tid < w)
#pragma unroll
      for (int k = 0; k < LOSS_SUMS; ++k) red[k][tid] += red[k][tid + w];
    __syncthreads();
  }
  if (tid == 0) {
    float n_linker = 0.f;                                    // numbers_of_nodes (edm.py:405-407): exact for a 0/1 mask
    for (int n = 0; n < N; ++n) n_linker += a.lm[(size_t)b * N + n];
    // x part of kl_prior, gaussian_kl_for_dimension (edm.py:450-463) with d = 3 * n_linker and p = N(0, 1):
    // d*log(1/sigma_T) + 0.5*(d*sigma_T^2 + ||mu_x||^2)/1 - 0.5*d
    const float dof = __fmul_rn(n_linker, 3.f);
    const float kl_x = __fsub_rn(__fadd_rn(__fmul_rn(dof, log_inv_sigma_T),
                                           __fmul_rn(0.5f, __fadd_rn(__fmul_rn(dof, sigma2_T), red[3][0]))),
                                 __fmul_rn(0.5f, dof));
    float* o = a.terms + (size_t)b * DL_LOSS_TERMS;
    o[DL_LOSS_ERROR_T] = red[0][0];
    o[DL_LOSS_NOISE] = sqrtf(red[2][0]);
    o[DL_LOSS_LOG_P_X] = __fmul_rn(-0.5f, red[1][0]);
    o[DL_LOSS_LOG_P_H] = red[5][0];
    o[DL_LOSS_KL_PRIOR] = __fadd_rn(kl_x, red[4][0]);
    o[DL_LOSS_N_LINKER] = n_linker;
  }
}

}  // namespace dl
