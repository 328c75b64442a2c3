// Long recordings: overlapping fixed-length windows, speaker alignment between neighbouring windows and crossfade
// stitching, all on the device.
//
// Geometry (window W samples, hop H, overlap O = W - H, W/2 <= H < W): a recording of T samples has
//   n = 1                       if T <= W
//   n = 1 + ceil((T - W) / H)   otherwise
// windows; window j covers [jH, jH + W), samples at or past T are zeros.  Windows of R recordings are flattened as
// w = r n + j.  Because H >= W/2 every sample lies in one or two windows, and because (n - 2) H + W < T every overlap
// [(j+1) H, j H + W) lies entirely below T, so the alignment statistics never see padding.
//
// No reference counterpart: the reference separates whole fixed-length clips (its training clips are 2 s).
#include <algorithm>

#include "common.cuh"

namespace vatss {

constexpr int LF_THREADS = 256;
constexpr int LF_NSUMS = 8;

int longform_windows(int T, int W, int H) {
  if (T <= W) return 1;
  return 1 + (int)(((long long)T - W + H - 1) / H);
}

// ---- cut -----------------------------------------------------------------------------------------------------------
// out (count, W): window first + blockIdx.y; zero past T
__global__ void __launch_bounds__(LF_THREADS)
k_window_cut(const float* __restrict__ mix, int T, int W, int H, int n, int first, float* __restrict__ out) {
  const int w = first + blockIdx.y;
  const int r = w / n, j = w - r * n;
  const long long start = (long long)j * H;
  const float* src = mix + (long long)r * T;
  float* dst = out + (long long)blockIdx.y * W;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < W; i += gridDim.x * blockDim.x) {
    const long long t = start + i;
    dst[i] = t < T ? src[t] : 0.f;
  }
}

// emb (R, E, Tv) -> out (count, E, Wv): window j takes frames [j Hv, j Hv + Wv), frames at or past Tv repeat Tv - 1.
// One CTA row per (window, feature) pair; blockIdx.z selects the speaker.
__global__ void __launch_bounds__(LF_THREADS)
k_window_cut_emb(const float* __restrict__ e1, const float* __restrict__ e2, int E, int Tv, int Wv, int Hv, int n,
                 int first, int count, float* __restrict__ o1, float* __restrict__ o2) {
  const float* src = blockIdx.z ? e2 : e1;
  float* dst = blockIdx.z ? o2 : o1;
  const long long rows = (long long)count * E;
  for (long long q = (long long)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); q < rows;
       q += (long long)gridDim.x * (blockDim.x / 32)) {
    const int wl = (int)(q / E), e = (int)(q - (long long)wl * E);
    const int w = first + wl;
    const int r = w / n, j = w - r * n;
    const float* s = src + ((long long)r * E + e) * Tv;
    float* d = dst + q * Wv;
    for (int f = threadIdx.x & 31; f < Wv; f += 32) d[f] = s[min(j * Hv + f, Tv - 1)];
  }
}

int launch_window_cut(const float* mix, const float* e1, const float* e2, int R, int T, int Tv, int E, int W, int H,
                      int spf, int first, int count, float* mix_out, float* e1_out, float* e2_out, cudaStream_t st) {
  const int n = longform_windows(T, W, H);
  if (count == 0) return 0;
  dim3 grid((unsigned)ceil_div(W, LF_THREADS * 4), (unsigned)count);
  k_window_cut<<<grid, LF_THREADS, 0, st>>>(mix, T, W, H, n, first, mix_out);
  VATSS_LAUNCH_OK();
  if (e1) {
    const long long rows = (long long)count * E;
    const int ctas = (int)std::min<long long>((rows + LF_THREADS / 32 - 1) / (LF_THREADS / 32), 1 << 16);
    k_window_cut_emb<<<dim3(ctas, 1, 2), LF_THREADS, 0, st>>>(e1, e2, E, Tv, W / spf, H / spf, n, first, count, e1_out,
                                                              e2_out);
    VATSS_LAUNCH_OK();
  }
  return 0;
}

// ---- alignment -----------------------------------------------------------------------------------------------------
// One CTA per adjacent pair (r, j), j < n - 1: over the overlap i in [0, O), a = window j at offset H + i, b = window
// j + 1 at offset i.  sums: [a1.b1, a1.b2, a2.b1, a2.b2, a1.a1, a2.a2, b1.b1, b2.b2] in fp64 with a fixed per-thread
// stride, a fixed shuffle tree and a fixed order over the warps, so the flags are bitwise reproducible.
__device__ __forceinline__ double lf_cos(double c, double ea, double eb) {
  return (ea > 0.0 && eb > 0.0) ? c / sqrt(ea * eb) : 0.0;
}

__global__ void __launch_bounds__(LF_THREADS)
k_stitch_corr(const float* __restrict__ y1, const float* __restrict__ y2, int n, int W, int H,
              uint8_t* __restrict__ flags, double* __restrict__ corr) {
  const int pair = blockIdx.x;
  const int r = pair / (n - 1), j = pair - r * (n - 1);
  const int O = W - H;
  const long long wa = ((long long)r * n + j) * W + H, wb = ((long long)r * n + j + 1) * W;
  double m[LF_NSUMS];
#pragma unroll
  for (int k = 0; k < LF_NSUMS; ++k) m[k] = 0.0;
  for (int i = threadIdx.x; i < O; i += LF_THREADS) {
    const double a1 = y1[wa + i], a2 = y2[wa + i], b1 = y1[wb + i], b2 = y2[wb + i];
    m[0] += a1 * b1; m[1] += a1 * b2; m[2] += a2 * b1; m[3] += a2 * b2;
    m[4] += a1 * a1; m[5] += a2 * a2; m[6] += b1 * b1; m[7] += b2 * b2;
  }
  __shared__ double red[LF_THREADS / 32][LF_NSUMS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < LF_NSUMS; ++k) {
    const double v = warp_sum_d(m[k]);
    if (lane == 0) red[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < LF_NSUMS) {
    double v = 0.0;
    for (int q = 0; q < LF_THREADS / 32; ++q) v += red[q][threadIdx.x];
    red[0][threadIdx.x] = v;   // each thread reads only its own column before overwriting it
    if (corr) corr[(long long)pair * LF_NSUMS + threadIdx.x] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const double* s = red[0];
    const double keep = lf_cos(s[0], s[4], s[6]) + lf_cos(s[3], s[5], s[7]);
    const double swap = lf_cos(s[1], s[4], s[7]) + lf_cos(s[2], s[5], s[6]);
    flags[pair] = swap > keep ? 1 : 0;
  }
}

// parity[r n + j] = flags[r (n-1) + 0] ^ ... ^ flags[r (n-1) + j - 1]: one warp per recording, 32 windows per step
__global__ void __launch_bounds__(LF_THREADS)
k_stitch_parity(const uint8_t* __restrict__ flags, int R, int n, uint8_t* __restrict__ parity) {
  const int r = blockIdx.x * (LF_THREADS / 32) + (threadIdx.x >> 5);
  if (r >= R) return;
  const int lane = threadIdx.x & 31;
  unsigned carry = 0;
  for (int j0 = 0; j0 < n; j0 += 32) {
    const int j = j0 + lane;
    // window j's parity is the XOR of the flags of pairs 0 .. j-1: lane takes pair j - 1
    const unsigned f = (j >= 1 && j < n) ? flags[(long long)r * (n - 1) + j - 1] : 0u;
    const unsigned mask = __ballot_sync(0xffffffffu, f != 0);
    const unsigned incl = mask & (0xffffffffu >> (31 - lane));
    if (j < n) parity[(long long)r * n + j] = (uint8_t)((carry ^ __popc(incl)) & 1u);
    carry ^= __popc(mask) & 1u;
  }
}

// out (R, T): the single covering window, or in an overlap i in [0, O) between windows j-1 and j
// (1 - a) y_{j-1}[H + i] + a y_j[i], a = (i + 0.5) / O.  Window j gives speaker s from its row s ^ parity_j.
__global__ void __launch_bounds__(LF_THREADS)
k_stitch_ola(const float* __restrict__ y1, const float* __restrict__ y2, const uint8_t* __restrict__ parity, int n,
             int T, int W, int H, float* __restrict__ s1, float* __restrict__ s2) {
  const int r = blockIdx.y;
  const int O = W - H;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < T; t += gridDim.x * blockDim.x) {
    const int j = min(t / H, n - 1);
    const int i = t - j * H;
    const long long w = (long long)r * n + j;
    const int p = parity[w];
    float o1 = (p ? y2 : y1)[w * W + i];
    float o2 = (p ? y1 : y2)[w * W + i];
    if (j > 0 && i < O) {
      const int q = parity[w - 1];
      const long long prev = (w - 1) * W + H + i;
      const float a = ((float)i + 0.5f) / (float)O;
      o1 = (1.0f - a) * (q ? y2 : y1)[prev] + a * o1;
      o2 = (1.0f - a) * (q ? y1 : y2)[prev] + a * o2;
    }
    s1[(long long)r * T + t] = o1;
    s2[(long long)r * T + t] = o2;
  }
}

static size_t round256(size_t b) { return (b + 255) / 256 * 256; }

size_t window_stitch_scratch_bytes(int R, int n) {
  if (R <= 0 || n <= 0) return 0;
  return round256((size_t)R * (n - 1) + 1) + round256((size_t)R * n);
}

int launch_window_stitch(const float* y1, const float* y2, int R, int T, int W, int H, float* s1, float* s2,
                         uint8_t* swaps_out, double* corr_out, void* scratch, cudaStream_t st) {
  const int n = longform_windows(T, W, H);
  uint8_t* flags = swaps_out ? swaps_out : reinterpret_cast<uint8_t*>(scratch);
  uint8_t* parity = reinterpret_cast<uint8_t*>(scratch) + round256((size_t)R * (n - 1) + 1);
  if (n > 1) {
    k_stitch_corr<<<R * (n - 1), LF_THREADS, 0, st>>>(y1, y2, n, W, H, flags, corr_out);
    VATSS_LAUNCH_OK();
  }
  k_stitch_parity<<<ceil_div(R, LF_THREADS / 32), LF_THREADS, 0, st>>>(flags, R, n, parity);
  VATSS_LAUNCH_OK();
  dim3 grid((unsigned)std::min(ceil_div(T, LF_THREADS * 4), 1 << 14), (unsigned)R);
  k_stitch_ola<<<grid, LF_THREADS, 0, st>>>(y1, y2, parity, n, T, W, H, s1, s2);
  VATSS_LAUNCH_OK();
  return 0;
}

}  // namespace vatss
