// GENERIC engine of the dual-path blocks: fp32 SIMT kernels for N <= 256, H <= 128 (multiple of 4) and
// head dim <= 64, at any sequence length (W_hh is held in fp16 for H >= 108, see launch_lstm_simt).
// They carry the small / odd configurations (the tiny golden fixtures, audio-only N=64 models
// until the tensor engine covers them) and are the on-device cross-check for the tcgen05
// TENSOR engine (tc_*.cu).  Semantics follow src/model/dptn.py:36-52 (TransformerDPRNN) and
// src/model/dprnn.py:24-47,65-89 (Intra/InterChunkRNN).
#include "common.cuh"

namespace vatss {

// ----------------------------------------------------------------------------------------
// C[M,Nout] = act(A[M,K]) * W[Nout,K]^T + bias (+bias2) (+ R)
// 64x64 tile, BK=16, 256 threads, 4x4 outputs per thread.
// ----------------------------------------------------------------------------------------
constexpr int GB_M = 64, GB_N = 64, GB_K = 16;

__global__ void __launch_bounds__(256)
k_gemm_simt(const float* __restrict__ A, long long lda, const float* __restrict__ W,
            const float* __restrict__ bias, const float* __restrict__ bias2, const float* __restrict__ R,
            long long ldr, float* __restrict__ Cout, long long ldc, long long M, int Nout, int K, int act,
            const float* __restrict__ prelu_a) {
  __shared__ float As[GB_K][GB_M + 4];
  __shared__ float Ws[GB_K][GB_N + 4];
  const long long m0 = (long long)blockIdx.x * GB_M;
  const int n0 = blockIdx.y * GB_N;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;  // tx -> n, ty -> m
  const float slope = (act == 2) ? prelu_a[0] : 0.f;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += GB_K) {
    // 64x16 tile of A and of W: 1024 elements each, 4 per thread; k is the fast index of the load
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int idx = tid + r * 256;
      const int kk = idx & 15, mm = idx >> 4;
      float a = 0.f, w = 0.f;
      if (m0 + mm < M && k0 + kk < K) {
        a = A[(m0 + mm) * lda + k0 + kk];
        if (act == 1) a = fmaxf(a, 0.f);
        else if (act == 2) a = a >= 0.f ? a : slope * a;
      }
      if (n0 + mm < Nout && k0 + kk < K) w = W[(size_t)(n0 + mm) * K + k0 + kk];
      As[kk][mm] = a;
      Ws[kk][mm] = w;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < GB_K; ++kk) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = Ws[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= Nout) continue;
      float v = acc[i][j];
      if (bias) v += bias[n];
      if (bias2) v += bias2[n];
      if (R) v += R[m * ldr + n];
      Cout[m * ldc + n] = v;
    }
  }
}

int launch_gemm_simt(const float* A, long long lda, const float* W, const float* bias, const float* bias2,
                     const float* R, long long ldr, float* Cout, long long ldc, long long M, int Nout, int K,
                     int act, const float* prelu_a, cudaStream_t st) {
  if (M == 0) return 0;
  dim3 grid(ceil_div(M, GB_M), ceil_div(Nout, GB_N));
  k_gemm_simt<<<grid, 256, 0, st>>>(A, lda, W, bias, bias2, R, ldr, Cout, ldc, M, Nout, K, act, prelu_a);
  VATSS_LAUNCH_OK();
  return 0;
}

// ----------------------------------------------------------------------------------------
// LayerNorm over the feature axis (biased variance, eps 1e-5), one warp per row.
//   mode 0: out = LN(in + res)      (DPTN: dptn.py:46-47,50-51)
//   mode 1: out = LN(in) + res      (DPRNN: dprnn.py:42-45)
// ----------------------------------------------------------------------------------------
constexpr int LN_MAX_NI = 8;

__global__ void __launch_bounds__(256)
k_layernorm(const float* __restrict__ in, const float* __restrict__ res, const float* __restrict__ w,
            const float* __restrict__ b, float* __restrict__ out, long long rows, int N, int mode) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int NI = (N + 31) / 32;
  float v[LN_MAX_NI];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAX_NI; ++i) {
    v[i] = 0.f;
    const int n = lane + 32 * i;
    if (i < NI && n < N) {
      float x = in[row * N + n];
      if (mode == 0 && res) x += res[row * N + n];
      v[i] = x;
      sum += x;
    }
  }
  const float mean = warp_sum(sum) / (float)N;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAX_NI; ++i) {
    const int n = lane + 32 * i;
    if (i < NI && n < N) {
      const float d = v[i] - mean;
      sq += d * d;
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / (float)N + 1e-5f);
#pragma unroll
  for (int i = 0; i < LN_MAX_NI; ++i) {
    const int n = lane + 32 * i;
    if (i < NI && n < N) {
      float y = (v[i] - mean) * rstd * w[n] + b[n];
      if (mode == 1 && res) y += res[row * N + n];
      out[row * N + n] = y;
    }
  }
}

int launch_layernorm(const float* in, const float* res, const float* w, const float* b, float* out,
                     long long rows, int N, int mode, cudaStream_t st) {
  VATSS_CHECK_ARG(N <= 32 * LN_MAX_NI, "layernorm: N=%d unsupported", N);
  if (rows == 0) return 0;
  k_layernorm<<<ceil_div(rows, 8), 256, 0, st>>>(in, res, w, b, out, rows, N, mode);
  VATSS_LAUNCH_OK();
  return 0;
}

// ----------------------------------------------------------------------------------------
// Multi-head self-attention core: out[row, h*hd:(h+1)*hd] = softmax(q k^T / sqrt(hd)) v
// qkv rows are (q | k | v), each N wide (nn.MultiheadAttention packed in_proj, dptn.py:16-21).
// One CTA per (sequence, head, block of 128 queries); one query per thread with an online
// softmax.  K and V of the head stream through shared memory in tiles of ATT_TILE_FLOATS / HDMAX
// keys, so any sequence length runs.  HDMAX is the register size of q and the accumulator: EXACT
// instances (hd = HDMAX, the powers of two) run unpredicated loops, the others take any runtime
// hd <= HDMAX (so every hd up to 64 runs).
// ----------------------------------------------------------------------------------------
constexpr int ATT_THREADS = 128;
constexpr int ATT_TILE_FLOATS = 4096;  // per operand: 16 KB of K and 16 KB of V

template <int HDMAX, bool EXACT>
__global__ void __launch_bounds__(ATT_THREADS)
k_attention_simt(const float* __restrict__ qkv, float* __restrict__ out, SeqMap map, int N, int hd_rt) {
  const int hd = EXACT ? HDMAX : hd_rt;
  constexpr int TILE = ATT_TILE_FLOATS / HDMAX;  // keys per tile
  __shared__ float sK[TILE * HDMAX];             // [TILE][HDMAX], columns >= hd unused
  __shared__ float sV[TILE * HDMAX];
  const int g = blockIdx.x, h = blockIdx.y;
  const int len = map.len;
  const int t = blockIdx.z * ATT_THREADS + threadIdx.x;
  const bool active = t < len;
  const long long r = active ? map.row(g, t) : 0;
  const float scale = rsqrtf((float)hd);
  float q[HDMAX], acc[HDMAX];
#pragma unroll
  for (int d = 0; d < HDMAX; ++d) {
    q[d] = (active && (EXACT || d < hd)) ? qkv[r * 3 * N + h * hd + d] * scale : 0.f;
    acc[d] = 0.f;
  }
  float m = -INFINITY, l = 0.f;
  for (int j0 = 0; j0 < len; j0 += TILE) {
    const int nk = min(TILE, len - j0);
    __syncthreads();  // the previous tile has been consumed
    for (int i = threadIdx.x; i < nk * hd; i += ATT_THREADS) {
      const int j = i / hd, d = i - j * hd;
      const long long rk = map.row(g, j0 + j);
      sK[j * HDMAX + d] = qkv[rk * 3 * N + N + h * hd + d];
      sV[j * HDMAX + d] = qkv[rk * 3 * N + 2 * N + h * hd + d];
    }
    __syncthreads();
    if (!active) continue;
    for (int j = 0; j < nk; ++j) {
      float s = 0.f;
#pragma unroll
      for (int d = 0; d < HDMAX; ++d)
        if (EXACT || d < hd) s = fmaf(q[d], sK[j * HDMAX + d], s);
      if (s > m) {
        const float c = expf(m - s);
        l *= c;
#pragma unroll
        for (int d = 0; d < HDMAX; ++d) acc[d] *= c;
        m = s;
      }
      const float p = expf(s - m);
      l += p;
#pragma unroll
      for (int d = 0; d < HDMAX; ++d)
        if (EXACT || d < hd) acc[d] = fmaf(p, sV[j * HDMAX + d], acc[d]);
    }
  }
  if (!active) return;
  const float inv = 1.f / l;
#pragma unroll
  for (int d = 0; d < HDMAX; ++d)
    if (EXACT || d < hd) out[r * N + h * hd + d] = acc[d] * inv;
}

template <int HDMAX, bool EXACT>
static int attention_launch(const float* qkv, float* out, SeqMap map, int N, int heads, cudaStream_t st) {
  VATSS_CHECK_ARG(heads <= 65535 && ceil_div(map.len, ATT_THREADS) <= 65535,
                  "attention: %d heads x length %d exceed the grid", heads, map.len);
  dim3 grid(map.G, heads, ceil_div(map.len, ATT_THREADS));
  k_attention_simt<HDMAX, EXACT><<<grid, ATT_THREADS, 0, st>>>(qkv, out, map, N, N / heads);
  VATSS_LAUNCH_OK();
  return 0;
}

int launch_attention_simt(const float* qkv, float* out, SeqMap map, int N, int heads, cudaStream_t st) {
  VATSS_CHECK_ARG(heads > 0 && N % heads == 0, "attention: N=%d not divisible by heads=%d", N, heads);
  const int hd = N / heads;
  VATSS_CHECK_ARG(hd <= 64, "attention: head dim %d unsupported by the generic kernel (max 64)", hd);
  if (map.G == 0 || map.len == 0) return 0;
  switch (hd) {
    case 1: return attention_launch<1, true>(qkv, out, map, N, heads, st);
    case 2: return attention_launch<2, true>(qkv, out, map, N, heads, st);
    case 4: return attention_launch<4, true>(qkv, out, map, N, heads, st);
    case 8: return attention_launch<8, true>(qkv, out, map, N, heads, st);
    case 16: return attention_launch<16, true>(qkv, out, map, N, heads, st);
    case 32: return attention_launch<32, true>(qkv, out, map, N, heads, st);
    case 64: return attention_launch<64, true>(qkv, out, map, N, heads, st);
    default: break;
  }
  if (hd < 8) return attention_launch<8, false>(qkv, out, map, N, heads, st);
  if (hd < 16) return attention_launch<16, false>(qkv, out, map, N, heads, st);
  if (hd < 32) return attention_launch<32, false>(qkv, out, map, N, heads, st);
  return attention_launch<64, false>(qkv, out, map, N, heads, st);
}

// ----------------------------------------------------------------------------------------
// LSTM recurrence (one layer, h0=c0=0, gate order i,f,g,o): nn.LSTM, dptn.py:23-29,49.
//   gates_t = pre[row(g,t)] + h_{t-1} Whh^T ; c = sig(f) c + sig(i) tanh(g) ; h = sig(o) tanh(c)
// `pre` already holds x W_ih^T + b_ih + b_hh.  One CTA owns LSTM_ST sequences of one
// direction for all time steps; Whh^T lives in shared memory for the whole kernel (fp32 for
// H <= 104, fp16 for H >= 108); thread j owns gate column j.
// ----------------------------------------------------------------------------------------
constexpr int LSTM_ST = 8;

template <typename WT>
__device__ __forceinline__ float w_to_float(WT w);
template <>
__device__ __forceinline__ float w_to_float<float>(float w) { return w; }
template <>
__device__ __forceinline__ float w_to_float<__half>(__half w) { return __half2float(w); }

template <typename WT>
__global__ void __launch_bounds__(512)
k_lstm_simt(const float* __restrict__ pre, const float* __restrict__ Whh_f, const float* __restrict__ Whh_r,
            float* __restrict__ out, SeqMap map, int H, int ndir) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int G4 = 4 * H;
  float* s_h = reinterpret_cast<float*>(smem_raw);          // [ST][H]
  float* s_c = s_h + LSTM_ST * H;                            // [ST][H]
  float* s_g = s_c + LSTM_ST * H;                            // [ST][4H]
  WT* s_w = reinterpret_cast<WT*>(s_g + LSTM_ST * G4);       // [H][4H]  (Whh transposed)
  const int dir = blockIdx.y;
  const float* Whh = dir == 0 ? Whh_f : Whh_r;
  const int g0 = blockIdx.x * LSTM_ST;
  const int nseq = min(LSTM_ST, map.G - g0);
  const int tid = threadIdx.x, nthr = blockDim.x;
  for (int i = tid; i < G4 * H; i += nthr) {
    const int j = i / H, k = i - j * H;  // Whh[j][k]
    s_w[k * G4 + j] = (WT)Whh[i];
  }
  for (int i = tid; i < LSTM_ST * H; i += nthr) {
    s_h[i] = 0.f;
    s_c[i] = 0.f;
  }
  __syncthreads();
  const int len = map.len;
  const int ldp = ndir * G4, ldo = ndir * H;
  for (int step = 0; step < len; ++step) {
    const int t = dir == 0 ? step : len - 1 - step;
    for (int j = tid; j < G4; j += nthr) {
      float acc[LSTM_ST];
#pragma unroll
      for (int s = 0; s < LSTM_ST; ++s)
        acc[s] = (s < nseq) ? pre[map.row(g0 + s, t) * ldp + dir * G4 + j] : 0.f;
      for (int k = 0; k < H; k += 4) {  // H % 4 == 0 (checked by the launcher)
        const float w0 = w_to_float<WT>(s_w[(k + 0) * G4 + j]);
        const float w1 = w_to_float<WT>(s_w[(k + 1) * G4 + j]);
        const float w2 = w_to_float<WT>(s_w[(k + 2) * G4 + j]);
        const float w3 = w_to_float<WT>(s_w[(k + 3) * G4 + j]);
#pragma unroll
        for (int s = 0; s < LSTM_ST; ++s) {
          const float4 hv = *reinterpret_cast<const float4*>(s_h + s * H + k);  // warp-wide broadcast
          acc[s] = fmaf(w0, hv.x, acc[s]);
          acc[s] = fmaf(w1, hv.y, acc[s]);
          acc[s] = fmaf(w2, hv.z, acc[s]);
          acc[s] = fmaf(w3, hv.w, acc[s]);
        }
      }
#pragma unroll
      for (int s = 0; s < LSTM_ST; ++s) s_g[s * G4 + j] = acc[s];
    }
    __syncthreads();
    for (int i = tid; i < nseq * H; i += nthr) {
      const int s = i / H, u = i - s * H;
      const float* gs = s_g + s * G4;
      const float ig = sigmoidf_precise(gs[u]);
      const float fg = sigmoidf_precise(gs[H + u]);
      const float gg = tanhf(gs[2 * H + u]);
      const float og = sigmoidf_precise(gs[3 * H + u]);
      const float c = fg * s_c[i] + ig * gg;
      const float h = og * tanhf(c);
      s_c[i] = c;
      s_h[i] = h;
      out[map.row(g0 + s, t) * ldo + dir * H + u] = h;
    }
    __syncthreads();
  }
}

int launch_lstm_simt(const float* pre, const float* Whh_f, const float* Whh_r, float* out, SeqMap map, int H,
                     int ndir, cudaStream_t st) {
  VATSS_CHECK_ARG(H >= 4 && H <= 128 && H % 4 == 0,
                  "lstm: hidden_dim %d unsupported by the generic kernel (multiple of 4, max 128)", H);
  if (map.G == 0) return 0;
  int threads = ((4 * H + 31) / 32) * 32;
  if (threads > 512) threads = 512;
  const size_t state = (size_t)(2 * LSTM_ST * H + LSTM_ST * 4 * H) * sizeof(float);
  const size_t w32 = (size_t)4 * H * H * sizeof(float);
  dim3 grid(ceil_div(map.G, LSTM_ST), ndir);
  // fp32 except W_hh in fp16 for H >= 108: W_hh^T stays fp32 in shared memory while 16H^2 + 192H <= 200 KB
  // (H <= 104); above that it is rounded to fp16 (relative error 2^-11 per weight), the rest stays fp32.
  if (state + w32 <= 200 * 1024) {
    VATSS_CUDA_OK(cudaFuncSetAttribute(k_lstm_simt<float>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(state + w32)));
    k_lstm_simt<float><<<grid, threads, state + w32, st>>>(pre, Whh_f, Whh_r, out, map, H, ndir);
  } else {
    const size_t w16 = w32 / 2;
    VATSS_CUDA_OK(cudaFuncSetAttribute(k_lstm_simt<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(state + w16)));
    k_lstm_simt<__half><<<grid, threads, state + w16, st>>>(pre, Whh_f, Whh_r, out, map, H, ndir);
  }
  VATSS_LAUNCH_OK();
  return 0;
}

}  // namespace vatss
