// PIT SI-SNR loss and SI-SNR / SI-SNRi metrics in one pass over the five waveforms.
//
// Reference: SiSNRLoss.forward src/loss/ss_losses.py:100-114 (zero-mean, no eps, -20 log10 of the
// power ratio, batch mean), BaseSSLoss.forward :10-26 (batch-level 2-permutation PIT),
// SS2BaseMetric.forward src/metrics/base_metric.py:41-60 and SISNRiMetric.__call__
// src/metrics/si_snri.py:12-30 (torchmetrics SI-SNR: zero-mean, eps = FLT_EPSILON, 10 log10).
//
// Stage 1 (HBM-bound): every CTA reads one chunk of one utterance of all five signals once and
// reduces 16 raw moments (5 sums, 5 square sums, 6 cross products) with warp shuffles, in fp64.
// Stage 2 (one CTA): combines the chunks, centres the moments algebraically
//   <p_c,g_c> = Spg - Sp Sg / T,  ||g_c||^2 = Sgg - Sg^2/T, ...
// and evaluates the per-utterance values, the batch means and both PIT decisions on the device,
// so the host needs a single small read instead of the reference's 4-6 `.item()` syncs.
#include <float.h>

#include "common.cuh"

namespace vatss {

constexpr int SISNR_CHUNK = 8192;
constexpr int SISNR_NM = 16;

int sisnr_chunks(int T) { return T <= 0 ? 1 : (T + SISNR_CHUNK - 1) / SISNR_CHUNK; }

__global__ void __launch_bounds__(256)
k_sisnr_moments(const float* __restrict__ s1p, const float* __restrict__ s2p, const float* __restrict__ s1,
                const float* __restrict__ s2, const float* __restrict__ mix, int T, int chunks,
                double* __restrict__ scratch) {
  const int b = blockIdx.y, ch = blockIdx.x;
  const int t0 = ch * SISNR_CHUNK;
  const int t1 = min(T, t0 + SISNR_CHUNK);
  const size_t base = (size_t)b * T;
  double m[SISNR_NM];
#pragma unroll
  for (int i = 0; i < SISNR_NM; ++i) m[i] = 0.0;
  for (int t = t0 + threadIdx.x; t < t1; t += blockDim.x) {
    const double a = s1p[base + t], c = s2p[base + t], x = s1[base + t], y = s2[base + t];
    const double z = mix ? (double)mix[base + t] : 0.0;
    m[0] += a; m[1] += c; m[2] += x; m[3] += y; m[4] += z;
    m[5] += a * a; m[6] += c * c; m[7] += x * x; m[8] += y * y; m[9] += z * z;
    m[10] += a * x;  // s1p.s1
    m[11] += c * y;  // s2p.s2
    m[12] += a * y;  // s1p.s2
    m[13] += c * x;  // s2p.s1
    m[14] += z * x;  // mix.s1
    m[15] += z * y;  // mix.s2
  }
  __shared__ double red[8][SISNR_NM];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < SISNR_NM; ++i) {
    const double v = warp_sum_d(m[i]);
    if (lane == 0) red[warp][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < SISNR_NM) {
    double v = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += red[w][threadIdx.x];
    scratch[((size_t)b * chunks + ch) * SISNR_NM + threadIdx.x] = v;
  }
}

struct PairMoments {
  double dot, pp, gg;  // centred <p,g>, ||p||^2, ||g||^2
};

__device__ __forceinline__ PairMoments centred(const double* m, int ip, int ig, int icross, double invT) {
  PairMoments r;
  r.dot = m[icross] - m[ip] * m[ig] * invT;
  r.pp = m[5 + ip] - m[ip] * m[ip] * invT;
  r.gg = m[5 + ig] - m[ig] * m[ig] * invT;
  return r;
}

// Residual power ||p_c - a g_c||^2 = pp - dot^2/gg of the eps-free loss, shared by the forward and the backward so that
// both see the same value.  For a near-exact estimate the cancellation of the raw-moment centring can make it zero or
// negative: the forward then reports -inf and the backward writes a zero gradient for that prediction.
__device__ __forceinline__ double loss_residual(const PairMoments& pm) { return pm.pp - pm.dot * pm.dot / pm.gg; }

__global__ void __launch_bounds__(256)
k_sisnr_finalize(const double* __restrict__ scratch, int B, int T, int chunks, int has_mix,
                 double* __restrict__ rows, double* __restrict__ rows_loss, double* __restrict__ summary) {
  const double invT = 1.0 / (double)T;
  const double eps = (double)FLT_EPSILON;
  // pairs: (pred index, target index, cross index)
  const int P_[6] = {0, 1, 0, 1, 4, 4};
  const int G_[6] = {2, 3, 3, 2, 2, 3};
  const int X_[6] = {10, 11, 12, 13, 14, 15};
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    double m[SISNR_NM];
    for (int i = 0; i < SISNR_NM; ++i) m[i] = 0.0;
    for (int c = 0; c < chunks; ++c)
      for (int i = 0; i < SISNR_NM; ++i) m[i] += scratch[((size_t)b * chunks + c) * SISNR_NM + i];
    for (int q = 0; q < 6; ++q) {
      if (q >= 4 && !has_mix) {
        rows[b * 6 + q] = 0.0;
        continue;
      }
      const PairMoments pm = centred(m, P_[q], G_[q], X_[q], invT);
      // torchmetrics form
      const double alpha = (pm.dot + eps) / (pm.gg + eps);
      const double sig = alpha * alpha * pm.gg;
      double noise = sig - 2.0 * alpha * pm.dot + pm.pp;
      if (noise < 0.0) noise = 0.0;
      rows[b * 6 + q] = 10.0 * log10((sig + eps) / (noise + eps));
      if (q < 4) {
        // reference loss form, no eps: signal = dot^2/gg, noise = pp - dot^2/gg
        const double s = pm.dot * pm.dot / pm.gg;
        double n = loss_residual(pm);
        if (n < 0.0) n = 0.0;   // perfect estimate: rounding may push the residual power below zero (-inf)
        rows_loss[b * 4 + q] = -20.0 * log10(s / n);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double mean_m[6] = {0, 0, 0, 0, 0, 0}, mean_l[4] = {0, 0, 0, 0};
    for (int b = 0; b < B; ++b) {
      for (int q = 0; q < 6; ++q) mean_m[q] += rows[b * 6 + q];
      for (int q = 0; q < 4; ++q) mean_l[q] += rows_loss[b * 4 + q];
    }
    for (int q = 0; q < 6; ++q) mean_m[q] /= (double)B;
    for (int q = 0; q < 4; ++q) mean_l[q] /= (double)B;
    const double l1 = (mean_l[0] + mean_l[1]) * 0.5, l2 = (mean_l[2] + mean_l[3]) * 0.5;
    const double s1 = (mean_m[0] + mean_m[1]) * 0.5, s2 = (mean_m[2] + mean_m[3]) * 0.5;
    const double sep = s1 > s2 ? s1 : s2;  // Python max(perm_1, perm_2)
    summary[0] = (l2 < l1) ? l2 : l1;
    summary[1] = l1;
    summary[2] = l2;
    summary[3] = sep;
    summary[4] = has_mix ? sep - (mean_m[4] + mean_m[5]) * 0.5 : 0.0;
    summary[5] = mean_m[4];
    summary[6] = mean_m[5];
    summary[7] = (double)B;
  }
}

int launch_pit_sisnr(const float* s1p, const float* s2p, const float* s1, const float* s2, const float* mix,
                     int B, int T, double* rows, double* rows_loss, double* summary, double* scratch,
                     cudaStream_t st) {
  VATSS_CHECK_ARG(B > 0 && T > 0, "pit_sisnr: empty batch (B=%d, T=%d)", B, T);
  VATSS_CHECK_ARG(B <= 65535, "pit_sisnr: batch of %d utterances (at most 65535)", B);
  const int chunks = sisnr_chunks(T);
  dim3 grid(chunks, B);
  k_sisnr_moments<<<grid, 256, 0, st>>>(s1p, s2p, s1, s2, mix, T, chunks, scratch);
  VATSS_LAUNCH_OK();
  k_sisnr_finalize<<<1, 256, 0, st>>>(scratch, B, T, chunks, mix != nullptr, rows, rows_loss, summary);
  VATSS_LAUNCH_OK();
  return 0;
}

int launch_sisnr_moments(const float* s1p, const float* s2p, const float* s1, const float* s2, const float* mix, int B,
                         int T, double* scratch, cudaStream_t st) {
  const int chunks = sisnr_chunks(T);
  k_sisnr_moments<<<dim3(chunks, B), 256, 0, st>>>(s1p, s2p, s1, s2, mix, T, chunks, scratch);
  VATSS_LAUNCH_OK();
  return 0;
}

// ------------------------------------------------------------------------------------------
// SI-SDR (torchmetrics' scale_invariant_signal_distortion_ratio, which src/metrics/si_sdr.py wraps; zero_mean=False by
// default) from the same raw moments: alpha = (<p,t> + eps) / (||t||^2 + eps), 10 log10((||alpha t||^2 + eps) /
// (||alpha t - p||^2 + eps)), eps = FLT_EPSILON, both norms expanded in fp64.  zero_mean = 1 centres the moments first
// (then the value is the SI-SNR of k_sisnr_finalize).  Rows 4, 5 are NaN without a mixture.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_sisdr_finalize(const double* __restrict__ scratch, int B, int T, int chunks, int has_mix, int zero_mean,
                 double* __restrict__ rows, double* __restrict__ summary) {
  const double invT = zero_mean ? 1.0 / (double)T : 0.0;   // 0: the raw moments
  const double eps = (double)FLT_EPSILON;
  const int P_[6] = {0, 1, 0, 1, 4, 4};
  const int G_[6] = {2, 3, 3, 2, 2, 3};
  const int X_[6] = {10, 11, 12, 13, 14, 15};
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    double m[SISNR_NM];
    for (int i = 0; i < SISNR_NM; ++i) m[i] = 0.0;
    for (int c = 0; c < chunks; ++c)
      for (int i = 0; i < SISNR_NM; ++i) m[i] += scratch[((size_t)b * chunks + c) * SISNR_NM + i];
    for (int q = 0; q < 6; ++q) {
      if (q >= 4 && !has_mix) {
        rows[b * 6 + q] = __longlong_as_double(0x7ff8000000000000ll);
        continue;
      }
      const PairMoments pm = centred(m, P_[q], G_[q], X_[q], invT);
      const double alpha = (pm.dot + eps) / (pm.gg + eps);
      const double sig = alpha * alpha * pm.gg;
      double noise = sig - 2.0 * alpha * pm.dot + pm.pp;
      if (noise < 0.0) noise = 0.0;
      rows[b * 6 + q] = 10.0 * log10((sig + eps) / (noise + eps));
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) pit_summary7(rows, B, has_mix, summary);
}

int launch_pit_sisdr(const float* s1p, const float* s2p, const float* s1, const float* s2, const float* mix, int B,
                     int T, int zero_mean, double* rows, double* summary, double* scratch, cudaStream_t st) {
  VATSS_CHECK_ARG(B > 0 && T > 0, "pit_sisdr: empty batch (B=%d, T=%d)", B, T);
  VATSS_CHECK_ARG(B <= 65535, "pit_sisdr: batch of %d utterances (at most 65535)", B);
  if (int rc = launch_sisnr_moments(s1p, s2p, s1, s2, mix, B, T, scratch, st)) return rc;
  k_sisdr_finalize<<<1, 256, 0, st>>>(scratch, B, T, sisnr_chunks(T), mix != nullptr, zero_mean, rows, summary);
  VATSS_LAUNCH_OK();
  return 0;
}

// ------------------------------------------------------------------------------------------
// Backward of the batch-level PIT loss with respect to the two predictions (first piece of the training step,
// src/trainer/trainer.py:46 `batch["loss"].backward()` through BaseSSLoss.forward src/loss/ss_losses.py:10-26).
//   L = (1 / 2B) sum_b [ l_b(p1, g_pi(1)) + l_b(p2, g_pi(2)) ],  l = -20 log10(||s||^2 / ||e||^2),  s = a g_c,  e = p_c - s
//   d l / d p = -(40 / ln 10) ( g_c / <g_c, p_c>  -  e / ||e||^2 )        (g_c and e are zero-mean: the centring Jacobian is I)
// pi is the permutation the forward chose for the WHOLE batch (summary[1], summary[2]); the per-row centred moments come
// from the forward's scratch (raw chunk sums), so the backward reads the four waveforms once and writes two gradients.
// A prediction whose residual power (loss_residual) is <= 0, where the forward reports -inf, gets a zero gradient.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_sisnr_loss_backward(const float* __restrict__ s1p, const float* __restrict__ s2p, const float* __restrict__ s1,
                      const float* __restrict__ s2, int B, int T, int chunks, const double* __restrict__ scratch,
                      const double* __restrict__ summary, const float* __restrict__ grad_out, float* __restrict__ g1,
                      float* __restrict__ g2) {
  const int b = blockIdx.y;
  __shared__ double m[SISNR_NM];
  if (threadIdx.x < SISNR_NM) {
    double v = 0.0;
    for (int c = 0; c < chunks; ++c) v += scratch[((size_t)b * chunks + c) * SISNR_NM + threadIdx.x];
    m[threadIdx.x] = v;
  }
  __syncthreads();
  const bool swap = summary[2] < summary[1];   // loss_perm_2 < loss_perm_1 (ss_losses.py:24)
  const double invT = 1.0 / (double)T;
  const double up = (grad_out ? (double)grad_out[0] : 1.0) * (-40.0 / 2.302585092994046) / (2.0 * (double)B);
  // prediction 1 pairs with s1 (cross 10) or s2 (cross 12); prediction 2 with s2 (11) or s1 (13)
  const PairMoments a = centred(m, 0, swap ? 3 : 2, swap ? 12 : 10, invT);
  const PairMoments c = centred(m, 1, swap ? 2 : 3, swap ? 13 : 11, invT);
  const double mp1 = m[0] * invT, mp2 = m[1] * invT, mg1 = m[swap ? 3 : 2] * invT, mg2 = m[swap ? 2 : 3] * invT;
  const double al1 = a.dot / a.gg, al2 = c.dot / c.gg;
  const double n1 = loss_residual(a), n2 = loss_residual(c);
  // the forward clamped a residual <= 0 and reported -inf: no descent direction, a zero gradient (NaN stays NaN)
  const float* t1 = swap ? s2 : s1;
  const float* t2 = swap ? s1 : s2;
  const size_t base = (size_t)b * T;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < T; t += gridDim.x * blockDim.x) {
    const double gc1 = (double)t1[base + t] - mg1, gc2 = (double)t2[base + t] - mg2;
    const double e1 = (double)s1p[base + t] - mp1 - al1 * gc1, e2 = (double)s2p[base + t] - mp2 - al2 * gc2;
    g1[base + t] = n1 <= 0.0 ? 0.0f : (float)(up * (gc1 / a.dot - e1 / n1));
    g2[base + t] = n2 <= 0.0 ? 0.0f : (float)(up * (gc2 / c.dot - e2 / n2));
  }
}

int launch_pit_sisnr_backward(const float* s1p, const float* s2p, const float* s1, const float* s2, int B, int T,
                              const double* scratch, const double* summary, const float* grad_out, float* g1, float* g2,
                              cudaStream_t st) {
  VATSS_CHECK_ARG(B > 0 && T > 0, "pit_sisnr_backward: empty batch (B=%d, T=%d)", B, T);
  VATSS_CHECK_ARG(B <= 65535, "pit_sisnr_backward: batch of %d utterances (at most 65535)", B);
  const int chunks = sisnr_chunks(T);
  int gx = (T + 256 * 8 - 1) / (256 * 8);
  if (gx < 1) gx = 1;
  dim3 grid(gx, B);
  k_sisnr_loss_backward<<<grid, 256, 0, st>>>(s1p, s2p, s1, s2, B, T, chunks, scratch, summary, grad_out, g1, g2);
  VATSS_LAUNCH_OK();
  return 0;
}

}  // namespace vatss
