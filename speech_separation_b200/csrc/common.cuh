// Shared helpers for the VAT-SS sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/vatss.h"

namespace vatss {

void set_error(const char* fmt, ...);

#define VATSS_CHECK_ARG(cond, ...)          \
  do {                                      \
    if (!(cond)) {                          \
      ::vatss::set_error(__VA_ARGS__);      \
      return -1;                            \
    }                                       \
  } while (0)

#define VATSS_CUDA_OK(expr)                                                              \
  do {                                                                                   \
    cudaError_t e__ = (expr);                                                            \
    if (e__ != cudaSuccess) {                                                            \
      ::vatss::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, \
                         __LINE__);                                                      \
      return -2;                                                                         \
    }                                                                                    \
  } while (0)

// every kernel launch is followed by this: checks the launch and counts it (vatss_launch_count)
void count_launch();
#define VATSS_LAUNCH_OK()               \
  do {                                  \
    ::vatss::count_launch();            \
    VATSS_CUDA_OK(cudaGetLastError());  \
  } while (0)

// optional per-stage device timing (vatss_profile_begin/end); no-ops unless enabled
enum Stage {
  ST_FRONTEND = 0, ST_QKV, ST_ATTENTION, ST_OUTPROJ_LN, ST_LSTM_INPUT, ST_LSTM_RECURRENT, ST_FFN_LN, ST_TAIL,
  ST_SISNR, ST_COUNT
};
void stage_begin(int stage, cudaStream_t st);
void stage_end(int stage, cudaStream_t st);
struct StageScope {
  int stage; cudaStream_t st;
  StageScope(int s, cudaStream_t t) : stage(s), st(t) { stage_begin(s, t); }
  ~StageScope() { stage_end(stage, st); }
};

// Function attributes (dynamic shared-memory limit) are per DEVICE: `PerDeviceOnce::first()` is true the first time it is
// asked on each device ordinal (a process may run models on cuda:0 and later on cuda:1).
struct PerDeviceOnce {
  unsigned long long mask[4] = {0, 0, 0, 0};   // 256 ordinals; launches of one model come from one host thread
  bool first() {
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 255;
    const unsigned long long bit = 1ull << (dev & 63);
    const bool f = !(mask[dev >> 6] & bit);
    mask[dev >> 6] |= bit;
    return f;
  }
};

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// How sequences of a dual-path sub-block map onto rows of a token-major (B,S,C,N) tensor.
//   intra: sequence (b,s), position k  -> row (b*S+s)*C + k
//   inter: sequence (b,k), position s  -> row (b*S+s)*C + k
// row(g,t) = (g / J) * per_batch + (g % J) * j_stride + t * t_stride
struct SeqMap {
  int G;          // number of sequences
  int len;        // positions per sequence
  int J;          // sequences per utterance
  long long per_batch;  // rows per utterance (S*C)
  int j_stride;
  int t_stride;
  __host__ __device__ inline long long row(int g, int t) const {
    return (long long)(g / J) * per_batch + (long long)(g % J) * j_stride + (long long)t * t_stride;
  }
};

static inline SeqMap intra_map(int B, int S, int C) {
  SeqMap m;
  m.G = B * S; m.len = C; m.J = S; m.per_batch = (long long)S * C; m.j_stride = C; m.t_stride = 1;
  return m;
}
static inline SeqMap inter_map(int B, int S, int C) {
  SeqMap m;
  m.G = B * C; m.len = S; m.J = C; m.per_batch = (long long)S * C; m.j_stride = 1; m.t_stride = C;
  return m;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float sigmoidf_precise(float x) { return 1.0f / (1.0f + expf(-x)); }

// ---- launchers implemented in the .cu files (all enqueue on `st`, return 0 or <0) ----

// frontend.cu
int launch_visual_compress(const float* emb1, const float* emb2, const float* Wv, const float* bv,
                           int B, int E, int Tv, int N, float* vis, cudaStream_t st);
int launch_encoder(const float* mix, const float* Wenc, const float* vis, const float* gate,
                   const float* vln_w, const float* vln_b, int B, int T, int Tv, int N, int K, int L,
                   int S, int C, int P, float* enc, float* seg, __half* seg16, cudaStream_t st,
                   __half* seg16lo = nullptr);
int launch_segment_cm(const float* x, int B, int N, int L, int C, int P, float* out, cudaStream_t st);
int launch_overlap_add_cm(const float* y, int B, int N, int S, int C, int P, float* out, cudaStream_t st);

// generic_block.cu
// C[M,Nout] = act(A[M,K]) * W[Nout,K]^T + bias (+ R).  act: 0 none, 1 relu, 2 prelu(*prelu_a)
int launch_gemm_simt(const float* A, long long lda, const float* W, const float* bias, const float* bias2,
                     const float* R, long long ldr, float* Cout, long long ldc, long long M, int Nout, int K,
                     int act, const float* prelu_a, cudaStream_t st);
// mode 0: out = LN(in + res); mode 1: out = LN(in) + res   (res may be NULL)
int launch_layernorm(const float* in, const float* res, const float* w, const float* b, float* out,
                     long long rows, int N, int mode, cudaStream_t st);
int launch_attention_simt(const float* qkv, float* out, SeqMap map, int N, int heads, cudaStream_t st);
// pre: (rows, ndir*4H) gate pre-activations incl. both biases; out: (rows, ndir*H)
int launch_lstm_simt(const float* pre, const float* Whh_f, const float* Whh_r, float* out, SeqMap map,
                     int H, int ndir, cudaStream_t st);

// tail.cu
int launch_ola_token_major(const float* y, int B, int S, int C, int P, int L, int W, float* ola, __half* ola16,
                           cudaStream_t st);
int launch_mask_combine(const float* t, const float* g, const float* enc, float* u, long long n, cudaStream_t st);
int launch_decoder(const float* u, const float* Wd, int B, int L, int N, int K, int T, float* proj,
                   float* wav, cudaStream_t st);
int launch_decoder_ola(const float* proj, int pitch, int B, int L, int K, int T, float* wav, cudaStream_t st);
int launch_fold_head(const float* Whead, const float* bhead, const float* Wd, int N, int K, float* wfold, float* wdT,
                     float* cfold, cudaStream_t st);
int launch_fold_spk(const float* wfold, const float* Wspk, const float* bspk, int N, int K, float* w2, float* c2,
                    cudaStream_t st);
int launch_tail_fused(const __half* px, const float* enc, const float* w2, const float* c2, const float* wdT,
                      const float* cfold, int B, int S, int C, int P, int L, int N, int K, float* proj, cudaStream_t st);

// sisnr.cu
int sisnr_chunks(int T);
int launch_pit_sisnr(const float* s1p, const float* s2p, const float* s1, const float* s2, const float* mix,
                     int B, int T, double* rows, double* rows_loss, double* summary, double* scratch,
                     cudaStream_t st);
int launch_pit_sisnr_backward(const float* s1p, const float* s2p, const float* s1, const float* s2, int B, int T,
                              const double* scratch, const double* summary, const float* grad_out, float* g1, float* g2,
                              cudaStream_t st);

// longform.cu
int longform_windows(int T, int W, int H);
size_t window_stitch_scratch_bytes(int R, int n);
int launch_window_cut(const float* mix, const float* e1, const float* e2, int R, int T, int Tv, int E, int W, int H,
                      int spf, int first, int count, float* mix_out, float* e1_out, float* e2_out, cudaStream_t st);
int launch_window_stitch(const float* y1, const float* y2, int R, int T, int W, int H, float* s1, float* s2,
                         uint8_t* swaps_out, double* corr_out, void* scratch, cudaStream_t st);

}  // namespace vatss
