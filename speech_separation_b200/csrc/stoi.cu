// STOI and extended STOI (ESTOI) of the four PIT pairings of a batch, all on the device.
//
// Reference: src/metrics/stoi.py wraps torchmetrics' ShortTimeObjectiveIntelligibility, which calls pystoi 0.4
// `stoi(target, preds, fs, extended)` on the host, one utterance at a time.  DESIGN.md §8 has the pipeline, the fp64
// restatement the tests compare against, precision and measured times.
//
// Rows are [s1p.s1, s2p.s2, s1p.s2, s2p.s1] (the row order of vatss_pit_sisnr).  The silent-frame mask depends on the
// clean target only, so utterance b has two masks (t = 0: s1, t = 1: s2) and six compacted signals, numbered
// 3 t + k with k = 0 the target itself, 1 s1p, 2 s2p.
//
//   k_stoi_filter    one CTA: the 256-tap Hann window (fp64) and, when fs != 10 kHz, the Kaiser-windowed sinc of
//                    pystoi's resample_oct in fp64 (power series I0, sinpi), normalised to sum 1, stored as fp32 p h.
//   k_stoi_resample  y[n] = p sum_m h[n q - m p + L] x[m]; input slab of a tile of outputs staged in shared memory,
//                    fp32 taps and accumulation in increasing m.
//   k_stoi_energy    one warp per 256-sample frame of each target: 20 log10(||w x_f|| + eps) in fp64.
//   k_stoi_frames    one CTA per (utterance, target): maximum, strict mask e > max - 40, ordered compaction of the
//                    kept frame indices (ballot + warp offsets, no atomics) and their count K.
//   k_stoi_bands     16 STFT frames of one compacted signal per CTA, gathered straight from the kept frames (each
//                    compacted sample has at most two), windowed, direct DFT over bins 7..218 against a shared
//                    twiddle table, |X|^2, one-third octave band sums, sqrt: envelopes (15, K - 1) in fp32.
//   k_stoi_corr      one CTA per (utterance, pairing): fp64 segment correlations with a fixed reduction order.
//   k_stoi_finalize  one CTA: batch-level PIT summary.
// Every sum has an order fixed by the utterance's own K, so results are bitwise reproducible and do not depend on
// which utterances share the batch.
#include <float.h>

#include "common.cuh"

namespace vatss {

constexpr int STOI_FS = 10000;
constexpr int STOI_FRAME = 256;
constexpr int STOI_HOP = 128;
constexpr int STOI_BANDS = 15;
constexpr int STOI_SEG = 30;
constexpr int STOI_BIN0 = 7;      // first and one-past-last DFT bin of the bands
constexpr int STOI_NBIN = 212;    // bins 7 .. 218
constexpr int STOI_THREADS = 256;
constexpr int STOI_FT = 16;       // STFT frames per CTA of k_stoi_bands
constexpr int STOI_ESEG = 32;     // segments per step of the extended correlation
constexpr int STOI_SMEM_MAX = 48 * 1024;
constexpr double STOI_DYN_RANGE = 40.0;

// pystoi `thirdoct(10000, 512, 15, 150)`: band i covers bins [edge[i], edge[i+1]) (tests/test_stoi.py pins the table)
__constant__ int c_stoi_edges[STOI_BANDS + 1] = {7, 9, 11, 14, 17, 22, 27, 34, 43, 55, 69, 87, 109, 138, 174, 219};

static long long gcd_ll(long long a, long long b) {
  while (b) { const long long t = a % b; a = b; b = t; }
  return a;
}
__host__ __device__ inline long long floor_div(long long a, long long b) {   // b > 0
  return a >= 0 ? a / b : -((-a + b - 1) / b);
}
static size_t round256(size_t b) { return (b + 255) / 256 * 256; }

// Everything the launches need, derived from (B, T, fs) on the host.
struct StoiGeom {
  bool resample;
  int p, q;                 // 10000 / fs reduced
  long long L;              // filter half length (2L + 1 taps)
  long long T10;            // samples at 10 kHz
  int F;                    // 256-sample frames at hop 128 of a 10 kHz signal
  int Fs;                   // envelope stride: at most F - 1 STFT frames
  int tile, span;           // outputs per resample CTA, staged input samples
  size_t off_taps, off_rs, off_energy, off_idx, off_K, off_env, off_win, bytes;
};

static int stoi_geometry(int B, int T, int fs, StoiGeom& g) {
  VATSS_CHECK_ARG(B > 0 && T > 0, "stoi: empty batch (B=%d, T=%d)", B, T);
  VATSS_CHECK_ARG(B <= 16383, "stoi: B=%d utterances out of range (at most 16383)", B);
  VATSS_CHECK_ARG(fs > 0 && fs <= 1000000, "stoi: sample rate fs=%d out of range (1 .. 1000000)", fs);
  const long long d = gcd_ll(STOI_FS, fs);
  g.p = (int)(STOI_FS / d);
  g.q = (int)(fs / d);
  g.resample = fs != STOI_FS;
  g.L = 0;
  if (g.resample) {
    // the same double operations as pystoi's resample_oct, so L is the same integer
    const double stop = 1.0 / (2.0 * (double)(g.p > g.q ? g.p : g.q));
    const double roll = stop / 10.0;
    g.L = (long long)ceil((60.0 - 8.0) / (28.714 * roll));
  }
  g.T10 = g.resample ? ((long long)T * g.p + g.q - 1) / g.q : T;
  VATSS_CHECK_ARG(g.T10 >= STOI_FRAME, "stoi: %d samples at %d Hz are %lld at 10 kHz, shorter than one %d-sample frame",
                  T, fs, g.T10, STOI_FRAME);
  const long long F = 1 + (g.T10 - STOI_FRAME) / STOI_HOP;
  VATSS_CHECK_ARG(F < (1ll << 30), "stoi: %lld frames per utterance out of range", F);
  g.F = (int)F;
  g.Fs = g.F > 1 ? g.F - 1 : 1;
  g.tile = 1024;
  g.span = 0;
  if (g.resample) {
    for (;;) {
      g.span = (int)(((long long)(g.tile - 1) * g.q + 2 * g.L) / g.p + 2);
      if ((size_t)g.span * sizeof(float) <= STOI_SMEM_MAX || g.tile <= 32) break;
      g.tile /= 2;
    }
    VATSS_CHECK_ARG((size_t)g.span * sizeof(float) <= STOI_SMEM_MAX,
                    "stoi: resampling %d Hz to 10 kHz needs %d staged samples per tile", fs, g.span);
  }
  size_t o = 0;
  g.off_win = o;    o += round256(STOI_FRAME * sizeof(double));
  g.off_taps = o;   o += g.resample ? round256((size_t)(2 * g.L + 1) * sizeof(float)) : 0;
  g.off_rs = o;     o += g.resample ? round256((size_t)B * 4 * g.T10 * sizeof(float)) : 0;
  g.off_energy = o; o += round256((size_t)B * 2 * g.F * sizeof(double));
  g.off_idx = o;    o += round256((size_t)B * 2 * g.F * sizeof(int));
  g.off_K = o;      o += round256((size_t)B * 2 * sizeof(int));
  g.off_env = o;    o += round256((size_t)B * 6 * STOI_BANDS * g.Fs * sizeof(float));
  g.bytes = o;
  return 0;
}

size_t stoi_workspace_bytes(int B, int T, int fs) {
  StoiGeom g;
  return stoi_geometry(B, T, fs, g) ? 0 : g.bytes;
}

// The four inputs of utterance b, at 10 kHz: sig 0 s1p, 1 s2p, 2 s1, 3 s2.
struct StoiSignals {
  const float *s0, *s1, *s2, *s3;   // named, not an array: a dynamic index would copy the parameter to local memory
  long long stride;                 // between utterances
  __device__ __forceinline__ const float* get(int b, int k) const {
    return (k == 0 ? s0 : k == 1 ? s1 : k == 2 ? s2 : s3) + (long long)b * stride;
  }
};

// ---- filter and window ---------------------------------------------------------------------------------------------
__device__ double stoi_i0(double x) {   // modified Bessel function of order 0: sum_k ((x/2)^k / k!)^2
  const double y = 0.25 * x * x;
  double t = 1.0, s = 1.0;
  for (int k = 1; k < 500; ++k) {
    t *= y / ((double)k * (double)k);
    s += t;
    if (t < s * 1e-17) break;
  }
  return s;
}

// np.kaiser(2L + 1, beta)[i] * 2 p stop * np.sinc(2 stop (i - L))
__device__ double stoi_tap(long long i, long long L, int p, double stop, double beta, double i0_beta) {
  const double r = (double)(i - L) / (double)L;
  const double kw = stoi_i0(beta * sqrt(fmax(0.0, 1.0 - r * r))) / i0_beta;
  const double x = 2.0 * stop * (double)(i - L);
  const double sinc = x == 0.0 ? 1.0 : sinpi(x) / (M_PI * x);
  return kw * 2.0 * (double)p * stop * sinc;
}

__global__ void __launch_bounds__(1024)
k_stoi_filter(int resample, int p, int q, long long L, double* __restrict__ win, float* __restrict__ taps) {
  // np.hanning(258)[1:-1]: 0.5 + 0.5 cos(pi n / 257), n = 2 (r + 1) - 257
  for (int r = threadIdx.x; r < STOI_FRAME; r += blockDim.x)
    win[r] = 0.5 + 0.5 * cospi((double)(2 * r + 2 - (STOI_FRAME + 1)) / (double)(STOI_FRAME + 1));
  if (!resample) return;
  const double stop = 1.0 / (2.0 * (double)(p > q ? p : q));
  const double beta = 0.1102 * (60.0 - 8.7);
  const double i0_beta = stoi_i0(beta);
  const long long n = 2 * L + 1;
  double s = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) s += stoi_tap(i, L, p, stop, beta, i0_beta);
  __shared__ double red[32];
  s = warp_sum_d(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  double sum = 0.0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) sum += red[w];
  const double scale = (double)p / sum;   // h / sum(h), times the p of the polyphase sum
  for (long long i = threadIdx.x; i < n; i += blockDim.x) taps[i] = (float)(stoi_tap(i, L, p, stop, beta, i0_beta) * scale);
}

// ---- resample ------------------------------------------------------------------------------------------------------
// grid (tiles, 4 B): blockIdx.y = 4 b + sig; out (B, 4, T10)
__global__ void __launch_bounds__(STOI_THREADS)
k_stoi_resample(const float* __restrict__ s1p, const float* __restrict__ s2p, const float* __restrict__ s1,
                const float* __restrict__ s2, int T, long long T10, int p, int q, long long L,
                const float* __restrict__ taps, int tile, int span, float* __restrict__ out) {
  extern __shared__ float xs[];
  const int sig = blockIdx.y & 3, b = blockIdx.y >> 2;
  const float* src = (sig == 0 ? s1p : sig == 1 ? s2p : sig == 2 ? s1 : s2) + (long long)b * T;
  const long long n0 = (long long)blockIdx.x * tile;
  const long long m_lo = floor_div(n0 * q - L + p - 1, p);   // first input sample of the tile's first output
  for (int i = threadIdx.x; i < span; i += blockDim.x) {
    const long long m = m_lo + i;
    xs[i] = (m >= 0 && m < T) ? src[m] : 0.f;
  }
  __syncthreads();
  float* dst = out + (long long)blockIdx.y * T10;
  for (int i = threadIdx.x; i < tile; i += blockDim.x) {
    const long long n = n0 + i;
    if (n >= T10) break;
    const long long nq = n * q;
    const long long m_a = floor_div(nq - L + p - 1, p), m_b = floor_div(nq + L, p);
    const float* xm = xs + (m_a - m_lo);
    const float* h = taps + (nq - m_a * p + L);
    float acc = 0.f;
    for (long long k = 0; k <= m_b - m_a; ++k) acc = fmaf(h[-k * p], xm[k], acc);
    dst[n] = acc;
  }
}

// ---- frame energies and the silent-frame mask -----------------------------------------------------------------------
// grid (ceil(F / 8), 2 B): blockIdx.y = 2 b + t, one warp per frame
__global__ void __launch_bounds__(STOI_THREADS)
k_stoi_energy(StoiSignals sg, int F, const double* __restrict__ win, double* __restrict__ energy) {
  const int t = blockIdx.y & 1, b = blockIdx.y >> 1;
  const int f = blockIdx.x * (STOI_THREADS / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (f >= F) return;
  const float* x = sg.get(b, 2 + t) + (long long)f * STOI_HOP;
  double s = 0.0;
#pragma unroll
  for (int r = lane; r < STOI_FRAME; r += 32) {
    const double v = win[r] * (double)x[r];
    s = fma(v, v, s);
  }
  s = warp_sum_d(s);
  if (lane == 0) energy[(long long)blockIdx.y * F + f] = 20.0 * log10(sqrt(s) + DBL_EPSILON);
}

// one CTA of 1024 threads per (b, t): idx[(2b + t) F + k] = k-th kept frame, K[2b + t] = count
__global__ void __launch_bounds__(1024)
k_stoi_frames(const double* __restrict__ energy, int F, int* __restrict__ idx, int* __restrict__ Kc,
              int* __restrict__ kept_out) {
  const double* e = energy + (long long)blockIdx.x * F;
  int* out = idx + (long long)blockIdx.x * F;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __shared__ double redm[32];
  __shared__ int woff[32], wtot;
  double mx = -INFINITY;
  for (int f = threadIdx.x; f < F; f += blockDim.x) mx = fmax(mx, e[f]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) redm[warp] = mx;
  __syncthreads();
  mx = redm[0];
  for (int w = 1; w < 32; ++w) mx = fmax(mx, redm[w]);
  const double thr = mx - STOI_DYN_RANGE;
  int carry = 0;
  for (int f0 = 0; f0 < F; f0 += 1024) {
    const int f = f0 + threadIdx.x;
    const bool keep = f < F && e[f] > thr;
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) woff[warp] = __popc(bal);   // 1024 threads: all 32 warps write their count
    __syncthreads();
    if (warp == 0) {
      const int v = woff[lane];
      int incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
      }
      woff[lane] = incl - v;
      if (lane == 31) wtot = incl;
    }
    __syncthreads();
    if (keep) out[carry + woff[warp] + __popc(bal & ((1u << lane) - 1u))] = f;
    carry += wtot;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    Kc[blockIdx.x] = carry;
    if (kept_out) kept_out[blockIdx.x] = carry;
  }
}

// ---- compacted STFT and band envelopes ------------------------------------------------------------------------------
// grid (ceil(Fs / FT), 6, B).  STFT frame i of the compacted signal covers compacted samples [128 i, 128 i + 256); its
// first half is kept frames i-1 (from offset 128) + i (from 0), its second half kept frames i (from 128) + i+1 (from 0),
// each windowed; the sum is windowed once more.  env ((6 b + s) 15 + band) Fs + i.
__global__ void __launch_bounds__(STOI_THREADS)
k_stoi_bands(StoiSignals sg, int F, int Fs, const double* __restrict__ win, const int* __restrict__ idx,
             const int* __restrict__ Kc, float* __restrict__ env) {
  const int b = blockIdx.z, s = blockIdx.y, t = s / 3, k = s - 3 * t;
  const int K = Kc[2 * b + t];
  const int i0 = blockIdx.x * STOI_FT;
  if (i0 >= K - 1) return;
  const float* x = k == 0 ? sg.get(b, 2 + t) : sg.get(b, k - 1);
  const int* kept = idx + (long long)(2 * b + t) * F;
  __shared__ float w[STOI_FRAME];
  __shared__ float cs[512 + 16], sn[512 + 16];                 // padded: entry m at m + m / 32
  __shared__ __align__(16) float buf[STOI_FRAME * STOI_FT];    // [sample][frame]
  __shared__ float pw[STOI_FT][STOI_NBIN];
  for (int r = threadIdx.x; r < STOI_FRAME; r += blockDim.x) w[r] = (float)win[r];
  for (int m = threadIdx.x; m < 512; m += blockDim.x) {
    double sv, cv;
    sincospi((double)m / 256.0, &sv, &cv);
    cs[m + (m >> 5)] = (float)cv;
    sn[m + (m >> 5)] = (float)sv;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < STOI_FRAME * STOI_FT; e += blockDim.x) {
    const int r = e & (STOI_FRAME - 1), f = e >> 8, i = i0 + f;
    float v = 0.f;
    if (i < K - 1) {
      const int h = r >> 7, rr = r & (STOI_HOP - 1);
      const int ka = i + h - 1, kb = i + h;   // kb <= K - 1 always
      const float va = ka >= 0 ? w[STOI_HOP + rr] * x[(long long)kept[ka] * STOI_HOP + STOI_HOP + rr] : 0.f;
      const float vb = w[rr] * x[(long long)kept[kb] * STOI_HOP + rr];
      v = (va + vb) * w[r];
    }
    buf[r * STOI_FT + f] = v;
  }
  __syncthreads();
  const int j = threadIdx.x;
  if (j < STOI_NBIN) {
    const int bin = STOI_BIN0 + j;
    float re[STOI_FT], im[STOI_FT];
#pragma unroll
    for (int f = 0; f < STOI_FT; ++f) re[f] = im[f] = 0.f;
    const float4* b4 = reinterpret_cast<const float4*>(buf);
    for (int n = 0; n < STOI_FRAME; ++n) {
      const int m = (bin * n) & 511;
      const float c = cs[m + (m >> 5)], sv = sn[m + (m >> 5)];
#pragma unroll
      for (int g = 0; g < STOI_FT / 4; ++g) {
        const float4 a = b4[n * (STOI_FT / 4) + g];
        re[4 * g + 0] = fmaf(a.x, c, re[4 * g + 0]); im[4 * g + 0] = fmaf(a.x, sv, im[4 * g + 0]);
        re[4 * g + 1] = fmaf(a.y, c, re[4 * g + 1]); im[4 * g + 1] = fmaf(a.y, sv, im[4 * g + 1]);
        re[4 * g + 2] = fmaf(a.z, c, re[4 * g + 2]); im[4 * g + 2] = fmaf(a.z, sv, im[4 * g + 2]);
        re[4 * g + 3] = fmaf(a.w, c, re[4 * g + 3]); im[4 * g + 3] = fmaf(a.w, sv, im[4 * g + 3]);
      }
    }
#pragma unroll
    for (int f = 0; f < STOI_FT; ++f) pw[f][j] = re[f] * re[f] + im[f] * im[f];
  }
  __syncthreads();
  float* dst = env + (long long)(6 * b + s) * STOI_BANDS * Fs;
  for (int e = threadIdx.x; e < STOI_FT * STOI_BANDS; e += blockDim.x) {
    const int band = e / STOI_FT, f = e - band * STOI_FT;
    if (i0 + f >= K - 1) continue;
    float acc = 0.f;
    for (int q = c_stoi_edges[band]; q < c_stoi_edges[band + 1]; ++q) acc += pw[f][q - STOI_BIN0];
    dst[(long long)band * Fs + i0 + f] = sqrtf(acc);
  }
}

// ---- correlations ---------------------------------------------------------------------------------------------------
// grid (4, B).  Pairing q: (target t, prediction signal k) = (0,1) (1,2) (1,1) (0,2).
__global__ void __launch_bounds__(STOI_THREADS)
k_stoi_corr(const float* __restrict__ env, const int* __restrict__ Kc, int Fs, int extended,
            double* __restrict__ rows) {
  const int q = blockIdx.x, b = blockIdx.y;
  const int t = (q == 1 || q == 2) ? 1 : 0, k = (q == 0 || q == 2) ? 1 : 2;
  const int frames = Kc[2 * b + t] - 1;
  if (frames < STOI_SEG) {
    if (threadIdx.x == 0) rows[4 * b + q] = 1e-5;
    return;
  }
  const int J = frames - STOI_SEG + 1;
  const float* X = env + (long long)(6 * b + 3 * t) * STOI_BANDS * Fs;
  const float* Y = env + (long long)(6 * b + 3 * t + k) * STOI_BANDS * Fs;
  const double eps = DBL_EPSILON;
  double acc = 0.0;
  if (!extended) {
    const double clip = 1.0 + 5.623413251903491;   // 1 + 10^(-BETA / 20), BETA = -15 dB
    for (long long it = threadIdx.x; it < (long long)STOI_BANDS * J; it += blockDim.x) {
      const int band = (int)(it / J), j = (int)(it - (long long)band * J);
      const float* xp = X + (long long)band * Fs + j;
      const float* yp = Y + (long long)band * Fs + j;
      float xv[STOI_SEG], yv[STOI_SEG];
      double sxx = 0.0, syy = 0.0;
#pragma unroll
      for (int f = 0; f < STOI_SEG; ++f) {
        xv[f] = xp[f];
        yv[f] = yp[f];
        sxx = fma((double)xv[f], (double)xv[f], sxx);
        syy = fma((double)yv[f], (double)yv[f], syy);
      }
      const double c = sqrt(sxx) / (sqrt(syy) + eps);
      double mx = 0.0, my = 0.0;
#pragma unroll
      for (int f = 0; f < STOI_SEG; ++f) {
        mx += (double)xv[f];
        my += fmin(c * (double)yv[f], (double)xv[f] * clip);
      }
      mx /= STOI_SEG;
      my /= STOI_SEG;
      double nx = 0.0, ny = 0.0, dot = 0.0;
#pragma unroll
      for (int f = 0; f < STOI_SEG; ++f) {
        const double a = (double)xv[f] - mx, d = fmin(c * (double)yv[f], (double)xv[f] * clip) - my;
        nx = fma(a, a, nx);
        ny = fma(d, d, ny);
        dot = fma(a, d, dot);
      }
      acc += dot / ((sqrt(nx) + eps) * (sqrt(ny) + eps));
    }
  } else {
    // a step of ESEG segments: row statistics (mean, 1 / (norm + eps) over the 30 frames) of every (segment, band),
    // then every (segment, frame) column: row-normalised values, column mean and norm over the bands, correlation
    __shared__ double st[4][STOI_ESEG][STOI_BANDS];
    for (int j0 = 0; j0 < J; j0 += STOI_ESEG) {
      for (int e = threadIdx.x; e < STOI_ESEG * STOI_BANDS; e += blockDim.x) {
        const int band = e / STOI_ESEG, sj = e - band * STOI_ESEG, j = j0 + sj;
        if (j >= J) continue;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const float* p = (u ? Y : X) + (long long)band * Fs + j;
          double m = 0.0;
          for (int f = 0; f < STOI_SEG; ++f) m += (double)p[f];
          m /= STOI_SEG;
          double n2 = 0.0;
          for (int f = 0; f < STOI_SEG; ++f) {
            const double a = (double)p[f] - m;
            n2 = fma(a, a, n2);
          }
          st[2 * u][sj][band] = m;
          st[2 * u + 1][sj][band] = 1.0 / (sqrt(n2) + eps);
        }
      }
      __syncthreads();
      for (int e = threadIdx.x; e < STOI_ESEG * STOI_SEG; e += blockDim.x) {
        const int f = e / STOI_ESEG, sj = e - f * STOI_ESEG, j = j0 + sj;
        if (j >= J) continue;
        double xr[STOI_BANDS], yr[STOI_BANDS], mx = 0.0, my = 0.0;
#pragma unroll
        for (int band = 0; band < STOI_BANDS; ++band) {
          xr[band] = ((double)X[(long long)band * Fs + j + f] - st[0][sj][band]) * st[1][sj][band];
          yr[band] = ((double)Y[(long long)band * Fs + j + f] - st[2][sj][band]) * st[3][sj][band];
          mx += xr[band];
          my += yr[band];
        }
        mx /= STOI_BANDS;
        my /= STOI_BANDS;
        double nx = 0.0, ny = 0.0, dot = 0.0;
#pragma unroll
        for (int band = 0; band < STOI_BANDS; ++band) {
          const double a = xr[band] - mx, d = yr[band] - my;
          nx = fma(a, a, nx);
          ny = fma(d, d, ny);
          dot = fma(a, d, dot);
        }
        acc += dot / ((sqrt(nx) + eps) * (sqrt(ny) + eps));
      }
      __syncthreads();
    }
  }
  __shared__ double red[STOI_THREADS / 32];
  acc = warp_sum_d(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < STOI_THREADS / 32; ++w) s += red[w];
    rows[4 * b + q] = extended ? s / STOI_SEG / (double)J : s / ((double)J * STOI_BANDS);
  }
}

// summary: [mean_b (row0 + row1) / 2, mean_b (row2 + row3) / 2, max of the two]
__global__ void k_stoi_finalize(const double* __restrict__ rows, int B, double* __restrict__ summary) {
  if (threadIdx.x != 0) return;
  double p1 = 0.0, p2 = 0.0;
  for (int b = 0; b < B; ++b) {
    p1 += (rows[4 * b] + rows[4 * b + 1]) * 0.5;
    p2 += (rows[4 * b + 2] + rows[4 * b + 3]) * 0.5;
  }
  p1 /= (double)B;
  p2 /= (double)B;
  summary[0] = p1;
  summary[1] = p2;
  summary[2] = p1 > p2 ? p1 : p2;   // Python max(perm_1, perm_2)
}

int launch_stoi(const float* s1p, const float* s2p, const float* s1, const float* s2, int B, int T, int fs,
                int extended, double* rows, int* kept_out, double* summary, void* workspace, size_t bytes,
                cudaStream_t st) {
  StoiGeom g;
  if (stoi_geometry(B, T, fs, g)) return -1;
  VATSS_CHECK_ARG(bytes >= g.bytes, "stoi: workspace too small: %zu bytes given, %zu needed", bytes, g.bytes);
  char* ws = reinterpret_cast<char*>(workspace);
  double* win = reinterpret_cast<double*>(ws + g.off_win);
  float* taps = reinterpret_cast<float*>(ws + g.off_taps);
  float* rs = reinterpret_cast<float*>(ws + g.off_rs);
  double* energy = reinterpret_cast<double*>(ws + g.off_energy);
  int* idx = reinterpret_cast<int*>(ws + g.off_idx);
  int* Kc = reinterpret_cast<int*>(ws + g.off_K);
  float* env = reinterpret_cast<float*>(ws + g.off_env);

  k_stoi_filter<<<1, 1024, 0, st>>>(g.resample, g.p, g.q, g.L, win, taps);
  VATSS_LAUNCH_OK();
  StoiSignals sg;
  if (g.resample) {
    const long long tiles = (g.T10 + g.tile - 1) / g.tile;
    VATSS_CHECK_ARG(tiles < (1ll << 31), "stoi: %lld resample tiles", tiles);
    k_stoi_resample<<<dim3((unsigned)tiles, 4 * B), STOI_THREADS, g.span * sizeof(float), st>>>(
        s1p, s2p, s1, s2, T, g.T10, g.p, g.q, g.L, taps, g.tile, g.span, rs);
    VATSS_LAUNCH_OK();
    sg.s0 = rs; sg.s1 = rs + g.T10; sg.s2 = rs + 2 * g.T10; sg.s3 = rs + 3 * g.T10;
    sg.stride = 4 * g.T10;
  } else {
    sg.s0 = s1p; sg.s1 = s2p; sg.s2 = s1; sg.s3 = s2;
    sg.stride = T;
  }
  k_stoi_energy<<<dim3(ceil_div(g.F, STOI_THREADS / 32), 2 * B), STOI_THREADS, 0, st>>>(sg, g.F, win, energy);
  VATSS_LAUNCH_OK();
  k_stoi_frames<<<2 * B, 1024, 0, st>>>(energy, g.F, idx, Kc, kept_out);
  VATSS_LAUNCH_OK();
  k_stoi_bands<<<dim3(ceil_div(g.Fs, STOI_FT), 6, B), STOI_THREADS, 0, st>>>(sg, g.F, g.Fs, win, idx, Kc, env);
  VATSS_LAUNCH_OK();
  k_stoi_corr<<<dim3(4, B), STOI_THREADS, 0, st>>>(env, Kc, g.Fs, extended, rows);
  VATSS_LAUNCH_OK();
  k_stoi_finalize<<<1, 32, 0, st>>>(rows, B, summary);
  VATSS_LAUNCH_OK();
  return 0;
}

}  // namespace vatss
