// BSS-eval SDR with a distortion filter of L taps (torchmetrics' signal_distortion_ratio on its direct-solve path) for
// the six pairings [s1p.s1, s2p.s2, s1p.s2, s2p.s1, mix.s1, mix.s2] of a batch, and the batch-level PIT summary.
//
// Per (prediction p, target t), in fp64: optionally remove the means, normalise both by max(||x||, 1e-6),
//   r[l] = sum_n t[n] t[n+l],  b[l] = sum_n t[n] p[n+l]   (l < L),  r[0] += load_diag,
// solve the symmetric Toeplitz system R x = b, coh = b.x, SDR = 10 log10(coh / (1 - coh)).
//
// Stage 1 (k_sisnr_moments, sisnr.cu): sums and square sums give the means and norms without another pass.
// Stage 2 (k_sdr_corr): the raw lag sums, directly (no FFT).  A CTA owns one target, one chunk of 512 lags and a fixed
//   range of n, stages the target and its four partners (the target itself, s1p, s2p, mix) in shared memory a tile at
//   a time and accumulates in registers; a thread owns 8 consecutive lags of one partner and slides an 8 + 8 sample
//   window, so 16 shared loads feed 64 fp64 FMAs.  The n ranges depend on T only, and the partials are reduced in a
//   fixed order: results are bitwise reproducible and independent of the other utterances of the batch.
// Stage 3 (k_sdr_solve, a CTA per utterance and target): reduces the partials, normalises, and runs the Levinson
//   recursion in fp64 once per target for its three right-hand sides (O(L^2) instead of a dense O(L^3) solve).
//   A prediction error <= 0 (an all-zero target, or a singular R without load_diag) makes that target's rows NaN.
// Stage 4 (k_sdr_finalize): the summary.
#include <float.h>

#include "common.cuh"

namespace vatss {

constexpr int SDR_THREADS = 256;
constexpr int SDR_TILE = 1024;            // samples of n staged per step
constexpr int SDR_LAGS = 512;             // lags per CTA
constexpr int SDR_R = 8;                  // consecutive lags per thread
constexpr int SDR_MAX_PARTS = 128;        // n ranges per (utterance, target, lag chunk)
constexpr int SDR_MAX_L = 2048;           // k_sdr_solve keeps 8 L doubles in shared memory
constexpr int SDR_NM = 16;                // moments per chunk (k_sisnr_moments)
// partner samples staged per tile, padded by one double every 8 so that lanes 8 lags apart hit different banks
constexpr int SDR_PSPAN = SDR_TILE + SDR_LAGS;
constexpr int SDR_PPAD = SDR_PSPAN / 8 * 9;
constexpr size_t SDR_CORR_SMEM = (size_t)(SDR_TILE + 4 * SDR_PPAD) * sizeof(double);
static_assert(SDR_LAGS / SDR_R * 4 == SDR_THREADS, "one thread per (partner, 8-lag block)");

struct SdrGeom {
  int L, chunks, lag_chunks, Lpad, tiles, tiles_per_part, parts;
  size_t off_part, bytes;
};

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

static int sdr_geometry(int B, int T, int L, SdrGeom& g) {
  VATSS_CHECK_ARG(B > 0 && T > 0, "sdr: empty batch (B=%d, T=%d)", B, T);
  VATSS_CHECK_ARG(B <= 65535, "sdr: batch of %d utterances (at most 65535)", B);
  VATSS_CHECK_ARG(L >= 1, "sdr: filter_length %d must be at least 1", L);
  VATSS_CHECK_ARG(L <= T, "sdr: filter_length %d longer than the signals (T=%d)", L, T);
  VATSS_CHECK_ARG(L <= SDR_MAX_L, "sdr: filter_length %d above %d", L, SDR_MAX_L);
  g.L = L;
  g.chunks = sisnr_chunks(T);
  g.lag_chunks = (L + SDR_LAGS - 1) / SDR_LAGS;
  g.Lpad = g.lag_chunks * SDR_LAGS;
  g.tiles = ceil_div(T, SDR_TILE);
  g.tiles_per_part = ceil_div(g.tiles, SDR_MAX_PARTS);
  g.parts = ceil_div(g.tiles, g.tiles_per_part);
  g.off_part = align256((size_t)B * g.chunks * SDR_NM * sizeof(double));
  g.bytes = g.off_part + align256((size_t)B * 2 * g.parts * 4 * g.Lpad * sizeof(double));
  return 0;
}

size_t sdr_workspace_bytes(int B, int T, int filter_length) {
  SdrGeom g;
  return sdr_geometry(B, T, filter_length, g) ? 0 : g.bytes;
}

// sum of moment i of utterance b over its chunks, in chunk order
__device__ __forceinline__ double moment(const double* scratch, int b, int chunks, int i) {
  double v = 0.0;
  for (int c = 0; c < chunks; ++c) v += scratch[((size_t)b * chunks + c) * SDR_NM + i];
  return v;
}

// grid (parts, 2 * lag_chunks, B).  Partner k of target g: 0 the target, 1 s1p, 2 s2p, 3 mix.
// part[(((b * 2 + g) * parts + part) * 4 + k) * Lpad + l] = sum over the part's n of t[n] p_k[n + l] (means removed
// first when zero_mean).
__global__ void __launch_bounds__(SDR_THREADS, 2)
k_sdr_corr(const float* __restrict__ s1p, const float* __restrict__ s2p, const float* __restrict__ s1,
           const float* __restrict__ s2, const float* __restrict__ mix, int T, int chunks, int tiles_per_part,
           int parts, int Lpad, int zero_mean, const double* __restrict__ moments, double* __restrict__ part) {
  extern __shared__ __align__(16) double sm[];
  double* ts = sm;                  // [SDR_TILE]
  double* ps = sm + SDR_TILE;       // [4][SDR_PPAD]
  const int p = blockIdx.x, g = blockIdx.y & 1, lc = blockIdx.y >> 1, b = blockIdx.z;
  const int nk = mix ? 4 : 3;
  const size_t base = (size_t)b * T;
  const float* tgt = g ? s2 : s1;
  const float* src[4] = {tgt, s1p, s2p, mix};
  __shared__ double mean[4];
  if (threadIdx.x < 4) {
    // moment index of the sum of each partner: s1p 0, s2p 1, s1 2, s2 3, mix 4
    const int mi[4] = {2 + g, 0, 1, 4};
    mean[threadIdx.x] = (zero_mean && (int)threadIdx.x < nk)
                            ? moment(moments, b, chunks, mi[threadIdx.x]) / (double)T : 0.0;
  }
  const int k = threadIdx.x / (SDR_LAGS / SDR_R), lb = threadIdx.x % (SDR_LAGS / SDR_R);
  const long long lag0 = (long long)lc * SDR_LAGS;
  double acc[SDR_R];
#pragma unroll
  for (int r = 0; r < SDR_R; ++r) acc[r] = 0.0;
  const int tile0 = p * tiles_per_part;
  const int tile1 = min(tile0 + tiles_per_part, (int)(((long long)T + SDR_TILE - 1) / SDR_TILE));
  for (int tile = tile0; tile < tile1; ++tile) {
    const long long n0 = (long long)tile * SDR_TILE;
    __syncthreads();   // mean[] written; the previous tile's readers are done
    for (int i = threadIdx.x; i < SDR_TILE; i += SDR_THREADS) {
      const long long n = n0 + i;
      ts[i] = n < T ? (double)tgt[base + n] - mean[0] : 0.0;
    }
    for (int kk = 0; kk < nk; ++kk) {
      const float* s = src[kk];
      const double mk = mean[kk];
      for (int x = threadIdx.x; x < SDR_PSPAN; x += SDR_THREADS) {
        const long long n = n0 + lag0 + x;
        ps[kk * SDR_PPAD + x + (x >> 3)] = n < T ? (double)s[base + n] - mk : 0.0;
      }
    }
    __syncthreads();
    if (k < nk) {
      // acc[r] += t[i] * p[i + 8 lb + r]; w holds p[i + 8 lb .. i + 8 lb + 15] (group j of 8 at padded offset 9 j)
      const double* pk = ps + k * SDR_PPAD;
      double w[2 * SDR_R];
#pragma unroll
      for (int q = 0; q < SDR_R; ++q) w[q] = pk[lb * 9 + q];
      for (int i = 0; i < SDR_TILE; i += SDR_R) {
        const int gi = (i >> 3) + lb + 1;
#pragma unroll
        for (int q = 0; q < SDR_R; ++q) w[SDR_R + q] = pk[gi * 9 + q];
        double tv[SDR_R];
#pragma unroll
        for (int u = 0; u < SDR_R; u += 2) {
          const double2 v = *reinterpret_cast<const double2*>(ts + i + u);
          tv[u] = v.x;
          tv[u + 1] = v.y;
        }
#pragma unroll
        for (int u = 0; u < SDR_R; ++u)
#pragma unroll
          for (int r = 0; r < SDR_R; ++r) acc[r] = fma(tv[u], w[u + r], acc[r]);
#pragma unroll
        for (int q = 0; q < SDR_R; ++q) w[q] = w[SDR_R + q];
      }
    }
  }
  if (k < nk) {
    double* out = part + ((((size_t)b * 2 + g) * parts + p) * 4 + k) * Lpad + lag0 + lb * SDR_R;
#pragma unroll
    for (int r = 0; r < SDR_R; ++r) out[r] = acc[r];
  }
}

// fixed-order block sum of 4 values; every thread gets the same result.  red: [SDR_THREADS / 32][4]
__device__ __forceinline__ void block_sum4(double v[4], double (*red)[4]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[i] = warp_sum_d(v[i]);
    if (lane == 0) red[warp][i] = v[i];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    double s = 0.0;
    for (int w = 0; w < SDR_THREADS / 32; ++w) s += red[w][i];
    v[i] = s;
  }
}

// grid (2, B): target g of utterance b.  Right-hand side j: 0 s1p, 1 s2p, 2 mix (partner j + 1 of k_sdr_corr).
__global__ void __launch_bounds__(SDR_THREADS)
k_sdr_solve(const double* __restrict__ moments, const double* __restrict__ part, int T, int chunks, int parts,
            int Lpad, int L, int has_mix, int zero_mean, double load_diag, double* __restrict__ rows) {
  extern __shared__ __align__(16) double sm[];
  double* r = sm;               // [L]  autocorrelation of the target
  double* rhs = sm + L;         // [3][L]
  double* x = sm + 4 * L;       // [3][L] solutions
  double* a = sm + 7 * L;       // [L] monic predictor, a[0] = 1
  __shared__ double red[SDR_THREADS / 32][4];
  __shared__ double nrm[4];     // target, s1p, s2p, mix: max(||x||, 1e-6)
  const int g = blockIdx.x, b = blockIdx.y;
  const int nj = has_mix ? 3 : 2;
  if (threadIdx.x < 4) {
    const int mi[4] = {2 + g, 0, 1, 4};
    const int i = mi[threadIdx.x];
    double ss = 0.0;
    if ((int)threadIdx.x <= nj) {
      ss = moment(moments, b, chunks, 5 + i);
      if (zero_mean) {
        const double s = moment(moments, b, chunks, i);
        ss -= s * s / (double)T;
      }
    }
    nrm[threadIdx.x] = fmax(sqrt(fmax(ss, 0.0)), 1e-6);
  }
  __syncthreads();
  const double* pb = part + (size_t)(b * 2 + g) * parts * 4 * Lpad;
  for (int l = threadIdx.x; l < L; l += SDR_THREADS) {
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    for (int q = 0; q < parts; ++q)
      for (int k = 0; k <= nj; ++k) s[k] += pb[((size_t)q * 4 + k) * Lpad + l];
    r[l] = s[0] / (nrm[0] * nrm[0]) + (l == 0 && load_diag >= 0.0 ? load_diag : 0.0);
    for (int j = 0; j < nj; ++j) {
      rhs[j * L + l] = s[j + 1] / (nrm[0] * nrm[j + 1]);
      x[j * L + l] = 0.0;
    }
    a[l] = l == 0 ? 1.0 : 0.0;
  }
  __syncthreads();
  double E = r[0];
  bool ok = E > 0.0;
  if (ok)
    for (int j = threadIdx.x; j < nj; j += SDR_THREADS) x[j * L] = rhs[j * L] / E;
  __syncthreads();
  for (int m = 1; m < L && ok; ++m) {
    // gamma = r[m] + sum_{j=1}^{m-1} a[j] r[m-j]; e_j = rhs_j[m] - sum_{i<m} r[m-i] x_j[i]
    double v[4] = {0.0, 0.0, 0.0, 0.0};
    for (int i = threadIdx.x; i < m; i += SDR_THREADS) {
      const double rr = r[m - i];
      v[0] = fma(a[i], rr, v[0]);   // a[0] = 1 gives the r[m] term
      for (int j = 0; j < nj; ++j) v[j + 1] = fma(rr, x[j * L + i], v[j + 1]);
    }
    block_sum4(v, red);
    const double kk = -v[0] / E;
    const double En = E * (1.0 - kk * kk);
    if (!(En > 0.0)) {
      ok = false;
      break;
    }
    // a <- a + kk * reverse(a) over 1..m-1 (pairs i, m-i), a[m] = kk
    for (int i = 1 + threadIdx.x; 2 * i <= m; i += SDR_THREADS) {
      const double ai = a[i], am = a[m - i];
      a[i] = fma(kk, am, ai);
      if (2 * i != m) a[m - i] = fma(kk, ai, am);
    }
    if (threadIdx.x == 0) a[m] = kk;
    __syncthreads();
    // x_j <- [x_j, 0] + (e_j / E_m) u, u[i] = a[m - i]
    for (int j = 0; j < nj; ++j) {
      const double mu = (rhs[j * L + m] - v[j + 1]) / En;
      for (int i = threadIdx.x; i <= m; i += SDR_THREADS) x[j * L + i] = fma(mu, a[m - i], x[j * L + i]);
    }
    E = En;
    __syncthreads();
  }
  __syncthreads();   // an early exit leaves threads still reading red[]
  // coherence b.x per right-hand side
  double v[4] = {0.0, 0.0, 0.0, 0.0};
  if (ok)
    for (int l = threadIdx.x; l < L; l += SDR_THREADS)
      for (int j = 0; j < nj; ++j) v[j] = fma(rhs[j * L + l], x[j * L + l], v[j]);
  block_sum4(v, red);
  if (threadIdx.x == 0) {
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    // row of (prediction j, target g): s1p.s1 0, s2p.s2 1, s1p.s2 2, s2p.s1 3, mix.s1 4, mix.s2 5
    const int q[3] = {g ? 2 : 0, g ? 1 : 3, 4 + g};
    for (int j = 0; j < 3; ++j)
      rows[6 * b + q[j]] = (ok && j < nj) ? 10.0 * log10(v[j] / (1.0 - v[j])) : nan;
  }
}

__global__ void k_sdr_finalize(const double* __restrict__ rows, int B, int has_mix, double* __restrict__ summary) {
  if (threadIdx.x == 0) pit_summary7(rows, B, has_mix, summary);
}

int launch_sdr(const float* s1p, const float* s2p, const float* s1, const float* s2, const float* mix, int B, int T,
               int filter_length, int zero_mean, double load_diag, double* rows, double* summary, void* workspace,
               size_t bytes, cudaStream_t st) {
  SdrGeom g;
  if (sdr_geometry(B, T, filter_length, g)) return -1;
  VATSS_CHECK_ARG(bytes >= g.bytes, "sdr: workspace too small: %zu bytes given, %zu needed", bytes, g.bytes);
  double* moments = reinterpret_cast<double*>(workspace);
  double* part = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + g.off_part);
  const size_t solve_smem = (size_t)8 * g.L * sizeof(double);
  static PerDeviceOnce once;
  if (once.first()) {
    VATSS_CUDA_OK(cudaFuncSetAttribute(k_sdr_corr, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SDR_CORR_SMEM));
    VATSS_CUDA_OK(cudaFuncSetAttribute(k_sdr_solve, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(8 * SDR_MAX_L * sizeof(double))));
  }
  if (int rc = launch_sisnr_moments(s1p, s2p, s1, s2, mix, B, T, moments, st)) return rc;
  k_sdr_corr<<<dim3(g.parts, 2 * g.lag_chunks, B), SDR_THREADS, SDR_CORR_SMEM, st>>>(
      s1p, s2p, s1, s2, mix, T, g.chunks, g.tiles_per_part, g.parts, g.Lpad, zero_mean, moments, part);
  VATSS_LAUNCH_OK();
  k_sdr_solve<<<dim3(2, B), SDR_THREADS, solve_smem, st>>>(moments, part, T, g.chunks, g.parts, g.Lpad, g.L,
                                                          mix != nullptr, zero_mean, load_diag, rows);
  VATSS_LAUNCH_OK();
  k_sdr_finalize<<<1, 32, 0, st>>>(rows, B, mix != nullptr, summary);
  VATSS_LAUNCH_OK();
  return 0;
}

}  // namespace vatss
