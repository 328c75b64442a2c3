// Separator tail: token-major overlap-add (+ centred pad), the masking head and the
// ConvTranspose1d decoder.  HBM-bound row-streaming kernels.
// Reference: src/model/dptn_wav.py:47-59,186-194; src/model/dptn.py:129-141,189;
//            src/model/dprnn.py:145-163.
#include <cstdlib>

#include "common.cuh"
#include "ptx.cuh"
#include "tc_kernels.cuh"

namespace vatss {

// ola[b,t,:] for t in [0,L): t' = t - padl; sum over chunks s with 0 <= t'-P*s < C of y[b,s,t'-P*s,:]
// (plain sum, increasing s), zero outside [0,(S-1)P+C).  W = row width (2N).
__global__ void __launch_bounds__(256)
k_ola_token_major(const float* __restrict__ y, int S, int C, int P, int L, int W4, int padl, int Lo,
                  long long total, float4* __restrict__ ola, uint2* __restrict__ ola16) {
  const float4* y4 = reinterpret_cast<const float4*>(y);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / W4;
    const int c = (int)(i - row * W4);
    const int b = (int)(row / L);
    const int t = (int)(row - (long long)b * L) - padl;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t >= 0 && t < Lo) {
      int s_lo = t - C + 1 + P - 1;
      s_lo = s_lo <= 0 ? 0 : s_lo / P;
      int s_hi = t / P;
      if (s_hi > S - 1) s_hi = S - 1;
      for (int s = s_lo; s <= s_hi; ++s) {
        const float4 v = y4[(((long long)b * S + s) * C + (t - P * s)) * W4 + c];
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
    }
    if (ola) ola[i] = acc;
    if (ola16) {
      const __half2 lo = __floats2half2_rn(acc.x, acc.y), hi = __floats2half2_rn(acc.z, acc.w);
      ola16[i] = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
    }
  }
}

int launch_ola_token_major(const float* y, int B, int S, int C, int P, int L, int W, float* ola, __half* ola16,
                           cudaStream_t st) {
  VATSS_CHECK_ARG(W % 4 == 0, "overlap-add: row width %d must be a multiple of 4", W);
  const int Lo = (S - 1) * P + C;
  const int padl = (L - Lo) / 2;
  const long long total = (long long)B * L * (W / 4);
  if (total == 0) return 0;
  int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  k_ola_token_major<<<blocks, 256, 0, st>>>(y, S, C, P, L, W / 4, padl, Lo, total,
                                            reinterpret_cast<float4*>(ola), reinterpret_cast<uint2*>(ola16));
  VATSS_LAUNCH_OK();
  return 0;
}


// ----------------------------------------------------------------------------------------
// Fused tail for the post-conv heads (dptn_wav.py:51-59,186-194; dprnn.py:269): everything between the speaker
// split and the decoder's overlap-add is linear per frame,
//   frames[b,l,spk,k] = sum_n Wd[n,k] (sum_m Whead[n,m] ola[b,l,spk*N+m] + bhead[n] + enc[b,l,n])
//                     = sum_m wfold[k,m] ola[...] + sum_n Wd[n,k] enc[b,l,n] + cfold[k],
// with wfold = Wd^T Whead and cfold = Wd^T bhead folded at weight-pack time (k_tail_fused below folds the speaker
// split in as well): the overlap-added tensor, the head output and their fp16 copies (2.4 GB of traffic) never exist.
// ----------------------------------------------------------------------------------------
__global__ void k_fold_head(const float* __restrict__ Whead, const float* __restrict__ bhead,
                            const float* __restrict__ Wd, int N, int K, float* __restrict__ wfold,
                            float* __restrict__ wdT, float* __restrict__ cfold) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < K * N) {
    const int k = i / N, m = i - k * N;
    double acc = 0.0;
    for (int n = 0; n < N; ++n) acc += (double)Wd[n * K + k] * (double)Whead[n * N + m];
    wfold[i] = (float)acc;
    wdT[i] = Wd[m * K + k];
  }
  if (i < K) {
    double acc = 0.0;
    for (int n = 0; n < N; ++n) acc += (double)Wd[n * K + i] * (double)bhead[n];
    cfold[i] = (float)acc;
  }
}

int launch_fold_head(const float* Whead, const float* bhead, const float* Wd, int N, int K, float* wfold, float* wdT,
                     float* cfold, cudaStream_t st) {
  k_fold_head<<<(K * N + 127) / 128, 128, 0, st>>>(Whead, bhead, Wd, N, K, wfold, wdT, cfold);
  VATSS_LAUNCH_OK();
  return 0;
}

// ----------------------------------------------------------------------------------------
// The speaker split is linear too (dptn_wav.py:47: Conv2d 1x1 on PReLU(x)), so it folds into the same pass:
//   frames[b,l,spk,k] = sum_n w2[spk,k,n] (sum over the <= 2 chunk rows of PReLU(x)[row, n])
//                       + rows * c2[spk,k] + sum_n Wd[n,k] enc[b,l,n] + cfold[k]
// with w2 = wfold Wspk[spk] and c2 = wfold bspk[spk].  The whole tail becomes one gather over the fp16 PReLU(x)
// copy (each token row is read exactly once) and the encoder output; the 1.4 GB speaker-split tensor never exists.
// ----------------------------------------------------------------------------------------
__global__ void k_fold_spk(const float* __restrict__ wfold, const float* __restrict__ Wspk,
                           const float* __restrict__ bspk, int N, int K, float* __restrict__ w2,
                           float* __restrict__ c2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 2 * K * N) {
    const int s = i / (K * N), k = (i / N) % K, n = i % N;
    double acc = 0.0;
    for (int m = 0; m < N; ++m) acc += (double)wfold[k * N + m] * (double)Wspk[(size_t)(s * N + m) * N + n];
    w2[i] = (float)acc;
  }
  if (i < 2 * K) {
    const int s = i / K, k = i % K;
    double acc = 0.0;
    for (int m = 0; m < N; ++m) acc += (double)wfold[k * N + m] * (double)bspk[s * N + m];
    c2[i] = (float)acc;
  }
}

int launch_fold_spk(const float* wfold, const float* Wspk, const float* bspk, int N, int K, float* w2, float* c2,
                    cudaStream_t st) {
  k_fold_spk<<<(2 * K * N + 127) / 128, 128, 0, st>>>(wfold, Wspk, bspk, N, K, w2, c2);
  VATSS_LAUNCH_OK();
  return 0;
}

// Round 2: the round-1 kernel (one frame per warp iteration, 2K full warp reductions of 5 shuffles each) moved 0.70 GB
// in 0.65 ms = 0.17 of the HBM roof: 16 resident warps per SM with 1 KB in flight each, and 2K x 10 shuffle / add
// instructions per frame.  Now every warp iteration covers FR = 4 consecutive frames with all of their gathers
// (FR x 3 row loads) issued before the first use, and the 2K per-lane partial sums are reduced by a TRANSPOSING
// butterfly: at step d a lane keeps the half of its values whose index bit matches its lane bit and receives the
// partner's partials of that half (16 -> 8 -> 4 -> 2 -> 1 values, 16 shuffles instead of 2K x 5); after five steps
// lane 2q holds output q.
template <int N, int K>
__global__ void __launch_bounds__(128)
k_tail_fused(const __half* __restrict__ px, const float* __restrict__ enc, const float* __restrict__ w2,
             const float* __restrict__ c2, const float* __restrict__ wdT, const float* __restrict__ cfold, int S, int C,
             int P, int L, int padl, int Lo, long long frames, float* __restrict__ proj) {
  constexpr int CH = N / 32;   // channels per lane (4 or 2)
  constexpr int FR = 4;        // frames per warp iteration
  static_assert(2 * K <= 16, "the transposing reduction carries 16 values");
  const int lane = threadIdx.x & 31, n0 = lane * CH;
  float wa[2][K][CH], wd[K][CH];
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      wa[0][k][i] = w2[k * N + n0 + i];
      wa[1][k][i] = w2[(K + k) * N + n0 + i];
      wd[k][i] = wdT[k * N + n0 + i];
    }
  // lane 2q (q < 2K) finally holds output q = (spk = q / K, tap q % K): its constants
  const int qout = lane >> 1;
  const bool owner = (lane & 1) == 0 && qout < 2 * K;
  const float cbias = owner ? c2[qout] : 0.f;
  const float cconst = owner ? cfold[qout % K] : 0.f;
  const long long warp0 = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long row0 = warp0 * FR; row0 < frames; row0 += nwarps * FR) {
    float o[FR][CH], e[FR][CH];
    int nrows[FR];
    // ---- all gathers of the FR frames first
#pragma unroll
    for (int f = 0; f < FR; ++f) {
      const long long row = row0 + f;
      nrows[f] = 0;
#pragma unroll
      for (int i = 0; i < CH; ++i) { o[f][i] = 0.f; e[f][i] = 0.f; }
      if (row < frames) {
        const int b = (int)(row / L);
        const int t = (int)(row - (long long)b * L) - padl;
        if constexpr (CH == 4) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(enc + row * N + n0));
          e[f][0] = v.x; e[f][1] = v.y; e[f][2] = v.z; e[f][3] = v.w;
        } else {
          const float2 v = __ldg(reinterpret_cast<const float2*>(enc + row * N + n0));
          e[f][0] = v.x; e[f][1] = v.y;
        }
        int s_lo = 0, s_hi = -1;
        if (t >= 0 && t < Lo) {
          s_lo = t - C + 1 + P - 1;
          s_lo = s_lo <= 0 ? 0 : s_lo / P;
          s_hi = t / P;
          if (s_hi > S - 1) s_hi = S - 1;
        }
        // s_lo > s_hi: a frame of the centred pad, or (step_size > chunk_size) a frame between two chunks that no
        // chunk covers - the reference's fold leaves it at zero, so nothing is loaded and no split bias is added
        if (s_lo <= s_hi) {
          nrows[f] = s_hi - s_lo + 1;
          // two rows for the 50 % overlap of the reference configs: both loads are issued unconditionally (the second
          // one re-reads the first row when there is only one) so that nothing depends on a data-dependent loop
          const bool two = s_hi > s_lo;
          const __half* src0 = px + (((long long)b * S + s_lo) * C + (t - P * s_lo)) * N + n0;
          const __half* src1 = two ? px + (((long long)b * S + s_lo + 1) * C + (t - P * (s_lo + 1))) * N + n0 : src0;
          const float w1 = two ? 1.f : 0.f;
          if constexpr (CH == 4) {
            const uint2 v0 = __ldg(reinterpret_cast<const uint2*>(src0));
            const uint2 v1 = __ldg(reinterpret_cast<const uint2*>(src1));
            const float2 a0 = __half22float2(*reinterpret_cast<const __half2*>(&v0.x));
            const float2 c0 = __half22float2(*reinterpret_cast<const __half2*>(&v0.y));
            const float2 a1 = __half22float2(*reinterpret_cast<const __half2*>(&v1.x));
            const float2 c1 = __half22float2(*reinterpret_cast<const __half2*>(&v1.y));
            o[f][0] = fmaf(w1, a1.x, a0.x); o[f][1] = fmaf(w1, a1.y, a0.y);
            o[f][2] = fmaf(w1, c1.x, c0.x); o[f][3] = fmaf(w1, c1.y, c0.y);
          } else {
            const float2 a0 = __half22float2(__ldg(reinterpret_cast<const __half2*>(src0)));
            const float2 a1 = __half22float2(__ldg(reinterpret_cast<const __half2*>(src1)));
            o[f][0] = fmaf(w1, a1.x, a0.x); o[f][1] = fmaf(w1, a1.y, a0.y);
          }
          for (int s = s_lo + 2; s <= s_hi; ++s) {       // (more than two rows only for overlaps above 50 %)
            const __half* src = px + (((long long)b * S + s) * C + (t - P * s)) * N + n0;
            if constexpr (CH == 4) {
              const uint2 v = __ldg(reinterpret_cast<const uint2*>(src));
              const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x));
              const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
              o[f][0] += a.x; o[f][1] += a.y; o[f][2] += c.x; o[f][3] += c.y;
            } else {
              const float2 a = __half22float2(*reinterpret_cast<const __half2*>(src));
              o[f][0] += a.x; o[f][1] += a.y;
            }
          }
        }
      }
    }
    // ---- per frame: per-lane partials of the 2K outputs, transposing butterfly, store
#pragma unroll
    for (int f = 0; f < FR; ++f) {
      float acc[16];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        float pe = 0.f, p0 = 0.f, p1 = 0.f;
#pragma unroll
        for (int i = 0; i < CH; ++i) {
          pe = fmaf(wd[k][i], e[f][i], pe);
          p0 = fmaf(wa[0][k][i], o[f][i], p0);
          p1 = fmaf(wa[1][k][i], o[f][i], p1);
        }
        acc[k] = p0 + pe;
        acc[K + k] = p1 + pe;
      }
#pragma unroll
      for (int k = 2 * K; k < 16; ++k) acc[k] = 0.f;
      // step d = 16, 8, 4, 2: keep the half selected by the lane bit, add the partner's partials of that half
#pragma unroll
      for (int h = 8; h >= 1; h >>= 1) {
        const bool up = (lane & (2 * h)) != 0;       // lane bit 4, 3, 2, 1
#pragma unroll
        for (int i = 0; i < h; ++i) {
          const float keep = up ? acc[h + i] : acc[i];
          const float send = up ? acc[i] : acc[h + i];
          acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2 * h);
        }
      }
      const float outv = acc[0] + __shfl_xor_sync(0xffffffffu, acc[0], 1);
      const long long row = row0 + f;
      if (owner && row < frames) proj[row * (2 * K) + qout] = outv + (float)nrows[f] * cbias + cconst;
    }
  }
}

// ----------------------------------------------------------------------------------------
// Staged form of k_tail_fused for the reference's 50 % overlap (C = 2 P).  k_tail_fused is latency-bound: its gathers
// hang off 168-register threads (12 warps per SM, ncu: 29 % issue activity, long-scoreboard stalls, 0.22 of the HBM
// roof).  Here the rows come through shared memory: a WORK UNIT is one hop of one utterance - the P frames
// t in [j P, (j + 1) P) - whose sources are three CONTIGUOUS row ranges (the encoder frames, rows [P, 2P) of chunk
// j - 1 and rows [0, P) of chunk j), fetched by a producer thread with three 1-D bulk copies (cp.async.bulk, mbarrier
// completion) into a two-stage ring while the eight compute warps work on the previous unit: same per-frame
// arithmetic as k_tail_fused (lane = 4 channels, folded weights in registers, transposing butterfly), no index
// arithmetic per frame.  Units j = -1 and j = S + 1 carry the frames of the centred pad (encoder term only).
// ----------------------------------------------------------------------------------------
#ifndef TS_WARPS_N
#define TS_WARPS_N 8
#endif
#ifndef TS_FR
#define TS_FR 4
#endif
constexpr int TS_WARPS = TS_WARPS_N;        // compute warps
constexpr int TS_THREADS = 32 * (TS_WARPS + 1);
constexpr int TS_STAGES = 2;

template <int N, int K>
__global__ void __launch_bounds__(TS_THREADS, 1)
k_tail_staged(const __half* __restrict__ px, const float* __restrict__ enc, const float* __restrict__ w2,
              const float* __restrict__ c2, const float* __restrict__ wdT, const float* __restrict__ cfold, int B, int S,
              int P, int L, int padl, float* __restrict__ proj) {
  using namespace ptx;
  constexpr int CH = N / 32;
  constexpr int FR = TS_FR;
  static_assert(2 * K <= 16, "the transposing reduction carries 16 values");
  extern __shared__ __align__(128) unsigned char smem[];
  const uint32_t enc_bytes = (uint32_t)P * N * 4, px_bytes = (uint32_t)P * N * 2;
  const uint32_t stage_bytes = enc_bytes + 2 * px_bytes;
  const uint32_t base = smem_u32(smem);
  const uint32_t bars = base + TS_STAGES * stage_bytes;      // full[TS_STAGES], empty[TS_STAGES]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C = 2 * P;
  const int upu = S + 3;                                      // units per utterance: j = -1 .. S + 1
  const long long units = (long long)B * upu;
  if (threadIdx.x == 0) {
    for (int s = 0; s < TS_STAGES; ++s) {
      mbar_init(bars + 8 * s, 1);
      mbar_init(bars + 8 * (TS_STAGES + s), TS_WARPS);
    }
    fence_mbar_init();
  }
  __syncthreads();
  // unit u -> utterance b, hop j, its frames [l0, l0 + F) and the offset `off` of the first one inside the hop
  auto unit_geometry = [&](long long u, int& b, int& j, int& l0, int& F, int& off) {
    b = (int)(u / upu);
    j = (int)(u - (long long)b * upu) - 1;
    const int lb = padl + j * P;
    l0 = lb < 0 ? 0 : lb;
    const int le = lb + P < L ? lb + P : L;
    F = le - l0;
    off = l0 - lb;
  };
  if (warp == TS_WARPS) {
    // ---------------------------------------------------------------- producer
    if (lane == 0) {
      int i = 0;
      for (long long u = blockIdx.x; u < units; u += gridDim.x, ++i) {
        const int s = i % TS_STAGES, ph = (i / TS_STAGES) & 1;
        int b, j, l0, F, off;
        unit_geometry(u, b, j, l0, F, off);
        mbar_wait(bars + 8 * (TS_STAGES + s), ph ^ 1);
        const bool lo_ok = j >= 1 && j <= S, hi_ok = j >= 0 && j <= S - 1;
        const uint32_t fe = (uint32_t)F * N * 4, fp = (uint32_t)F * N * 2;
        const uint32_t dst = base + s * stage_bytes;
        mbar_expect_tx(bars + 8 * s, F > 0 ? fe + (lo_ok ? fp : 0) + (hi_ok ? fp : 0) : 0);
        if (F > 0) {
          bulk_load_1d(dst, enc + ((long long)b * L + l0) * N, fe, bars + 8 * s);
          if (lo_ok) bulk_load_1d(dst + enc_bytes, px + (((long long)b * S + j - 1) * C + P + off) * N, fp, bars + 8 * s);
          if (hi_ok) bulk_load_1d(dst + enc_bytes + px_bytes, px + (((long long)b * S + j) * C + off) * N, fp, bars + 8 * s);
        }
      }
    }
    return;
  }
  // ------------------------------------------------------------------ compute warps
  const int n0 = lane * CH;
  float wa[2][K][CH], wd[K][CH];
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      wa[0][k][i] = w2[k * N + n0 + i];
      wa[1][k][i] = w2[(K + k) * N + n0 + i];
      wd[k][i] = wdT[k * N + n0 + i];
    }
  const int qout = lane >> 1;
  const bool owner = (lane & 1) == 0 && qout < 2 * K;
  const float cbias = owner ? c2[qout] : 0.f;
  const float cconst = owner ? cfold[qout % K] : 0.f;
  int it = 0;
  for (long long u = blockIdx.x; u < units; u += gridDim.x, ++it) {
    const int s = it % TS_STAGES, ph = (it / TS_STAGES) & 1;
    int b, j, l0, F, off;
    unit_geometry(u, b, j, l0, F, off);
    const bool lo_ok = j >= 1 && j <= S, hi_ok = j >= 0 && j <= S - 1;
    const float nrows = (float)((lo_ok ? 1 : 0) + (hi_ok ? 1 : 0));
    const unsigned char* st = smem + s * stage_bytes;
    const float* sE = reinterpret_cast<const float*>(st);
    const __half* sLo = reinterpret_cast<const __half*>(st + enc_bytes);
    const __half* sHi = reinterpret_cast<const __half*>(st + enc_bytes + px_bytes);
    mbar_wait(bars + 8 * s, ph);
    // groups of FR frames, dealt round-robin with a per-unit rotation so that no warp always gets the extra group
    const int ngroups = (F + FR - 1) / FR;
    for (int g = (warp + it * 3) % TS_WARPS; g < ngroups; g += TS_WARPS) {
      float o[FR][CH], e[FR][CH];
#pragma unroll
      for (int f = 0; f < FR; ++f) {
        const int fi = g * FR + f;
#pragma unroll
        for (int i = 0; i < CH; ++i) { o[f][i] = 0.f; e[f][i] = 0.f; }
        if (fi < F) {
          if constexpr (CH == 4) {
            const float4 v = *reinterpret_cast<const float4*>(sE + fi * N + n0);
            e[f][0] = v.x; e[f][1] = v.y; e[f][2] = v.z; e[f][3] = v.w;
            if (lo_ok) {
              const uint2 r = *reinterpret_cast<const uint2*>(sLo + fi * N + n0);
              const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x));
              const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
              o[f][0] = a.x; o[f][1] = a.y; o[f][2] = c.x; o[f][3] = c.y;
            }
            if (hi_ok) {
              const uint2 r = *reinterpret_cast<const uint2*>(sHi + fi * N + n0);
              const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x));
              const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
              o[f][0] += a.x; o[f][1] += a.y; o[f][2] += c.x; o[f][3] += c.y;
            }
          } else {
            const float2 v = *reinterpret_cast<const float2*>(sE + fi * N + n0);
            e[f][0] = v.x; e[f][1] = v.y;
            if (lo_ok) {
              const float2 a = __half22float2(*reinterpret_cast<const __half2*>(sLo + fi * N + n0));
              o[f][0] = a.x; o[f][1] = a.y;
            }
            if (hi_ok) {
              const float2 a = __half22float2(*reinterpret_cast<const __half2*>(sHi + fi * N + n0));
              o[f][0] += a.x; o[f][1] += a.y;
            }
          }
        }
      }
#pragma unroll
      for (int f = 0; f < FR; ++f) {
        float acc[16];
#pragma unroll
        for (int k = 0; k < K; ++k) {
          float pe = 0.f, p0 = 0.f, p1 = 0.f;
#pragma unroll
          for (int i = 0; i < CH; ++i) {
            pe = fmaf(wd[k][i], e[f][i], pe);
            p0 = fmaf(wa[0][k][i], o[f][i], p0);
            p1 = fmaf(wa[1][k][i], o[f][i], p1);
          }
          acc[k] = p0 + pe;
          acc[K + k] = p1 + pe;
        }
#pragma unroll
        for (int k = 2 * K; k < 16; ++k) acc[k] = 0.f;
#pragma unroll
        for (int h = 8; h >= 1; h >>= 1) {
          const bool up = (lane & (2 * h)) != 0;
#pragma unroll
          for (int i = 0; i < h; ++i) {
            const float keep = up ? acc[h + i] : acc[i];
            const float send = up ? acc[i] : acc[h + i];
            acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2 * h);
          }
        }
        const float outv = acc[0] + __shfl_xor_sync(0xffffffffu, acc[0], 1);
        const int fi = g * FR + f;
        if (owner && fi < F) proj[((long long)b * L + l0 + fi) * (2 * K) + qout] = outv + nrows * cbias + cconst;
      }
    }
    // the stage was written by the async proxy and read with ordinary loads: order those reads before the bulk copy
    // that the arrival allows (DESIGN.md 3.4b)
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) mbar_arrive(bars + 8 * (TS_STAGES + s));   // this warp has finished reading the stage
  }
}

int g_tail_staged = -1;   // -1: VATSS_TAIL_STAGED from the environment (default 1); 0 keeps the gather kernel (cross-check)

// whole tail after the last dual-path block for the post-conv heads; returns 1 when (N, K) has no instance
int launch_tail_fused(const __half* px, const float* enc, const float* w2, const float* c2, const float* wdT,
                      const float* cfold, int B, int S, int C, int P, int L, int N, int K, float* proj, cudaStream_t st) {
  const long long frames = (long long)B * L;
  if (frames == 0) return 0;
  const int Lo = (S - 1) * P + C;
  const int padl = (L - Lo) / 2;
  // staged kernel: 50 % overlap, the centred pad fits one hop on either side, the ring fits shared memory
  {
    if (g_tail_staged < 0) { const char* e = getenv("VATSS_TAIL_STAGED"); g_tail_staged = e ? atoi(e) : 1; }
    const int staged_on = g_tail_staged;
    const size_t ring = (size_t)TS_STAGES * P * N * 8 + 64;
    if (staged_on && C == 2 * P && padl >= 0 && padl <= P && L - padl - Lo >= 0 && L - padl - Lo <= P &&
        ring <= 200 * 1024 && (P * N) % 8 == 0) {
      const long long units = (long long)B * (S + 3);
      const int grid = (int)(units < num_sms() ? units : num_sms());
#define VATSS_TAIL_STAGED(NN, KK)                                                                                     \
      if (N == NN && K == KK) {                                                                                       \
        static PerDeviceOnce configured;                                                                              \
        if (configured.first())                                                                                       \
          VATSS_CUDA_OK(cudaFuncSetAttribute(k_tail_staged<NN, KK>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                                             200 * 1024));                                                            \
        k_tail_staged<NN, KK><<<grid, TS_THREADS, ring, st>>>(px, enc, w2, c2, wdT, cfold, B, S, P, L, padl, proj);   \
        VATSS_LAUNCH_OK();                                                                                            \
        return 0;                                                                                                     \
      }
      VATSS_TAIL_STAGED(128, 7)
      VATSS_TAIL_STAGED(64, 7)
      VATSS_TAIL_STAGED(64, 2)
      VATSS_TAIL_STAGED(128, 2)
#undef VATSS_TAIL_STAGED
    }
  }
  const int blocks = (int)(ceil_div(frames, 16) < 148 * 12 ? ceil_div(frames, 16) : 148 * 12);
#define VATSS_TAIL_FUSED(NN, KK)                                                                                      \
  if (N == NN && K == KK) {                                                                                           \
    k_tail_fused<NN, KK><<<blocks, 128, 0, st>>>(px, enc, w2, c2, wdT, cfold, S, C, P, L, padl, Lo, frames, proj);    \
    VATSS_LAUNCH_OK();                                                                                                \
    return 0;                                                                                                         \
  }
  VATSS_TAIL_FUSED(128, 7)
  VATSS_TAIL_FUSED(64, 7)
  VATSS_TAIL_FUSED(64, 2)
  VATSS_TAIL_FUSED(128, 2)
#undef VATSS_TAIL_FUSED
  return 1;
}

// masking head (dptn.py:103-115,141,189): u = ReLU(tanh(t) * sigmoid(g)) * enc
__global__ void k_mask_combine(const float* __restrict__ t, const float* __restrict__ g,
                               const float* __restrict__ enc, float* __restrict__ u, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    const float m = tanhf(t[i]) * sigmoidf_precise(g[i]);
    u[i] = fmaxf(m, 0.f) * enc[i];
  }
}

int launch_mask_combine(const float* t, const float* g, const float* enc, float* u, long long n,
                        cudaStream_t st) {
  if (n == 0) return 0;
  int blocks = (int)((n + 255) / 256 < 148 * 16 ? (n + 255) / 256 : 148 * 16);
  k_mask_combine<<<blocks, 256, 0, st>>>(t, g, enc, u, n);
  VATSS_LAUNCH_OK();
  return 0;
}

// decoder stage 1: proj[b,l,k] = sum_n Wd[n,k] u[b,l,n]      (one warp per frame)
constexpr int DEC_MAX_K = 16;
__global__ void __launch_bounds__(256)
k_decoder_proj(const float* __restrict__ u, const float* __restrict__ Wd, long long rows, int N, int K,
               float* __restrict__ proj) {
  extern __shared__ float s_w[];  // [N][K]
  for (int i = threadIdx.x; i < N * K; i += blockDim.x) s_w[i] = Wd[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  float acc[DEC_MAX_K];
#pragma unroll
  for (int k = 0; k < DEC_MAX_K; ++k) acc[k] = 0.f;
  for (int n = lane; n < N; n += 32) {
    const float x = u[row * N + n];
#pragma unroll
    for (int k = 0; k < DEC_MAX_K; ++k)
      if (k < K) acc[k] = fmaf(s_w[n * K + k], x, acc[k]);
  }
#pragma unroll
  for (int k = 0; k < DEC_MAX_K; ++k)
    if (k < K) {
      const float v = warp_sum(acc[k]);
      if (lane == 0) proj[row * K + k] = v;
    }
}

// decoder stage 2: wav[b,i] = sum_{(l,k): st*l+k = i-padl} proj[b,l,k], zero outside (centred pad)
__global__ void k_decoder_ola(const float* __restrict__ proj, int pitch, int L, int K, int st, int T, int padl,
                              long long total, float* __restrict__ wav) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / T);
    const int j = (int)(i - (long long)b * T) - padl;
    float acc = 0.f;
    if (j >= 0 && j < (L - 1) * st + K) {
      // frames l with 0 <= j - st*l < K
      int l_lo = j - K + 1 + st - 1;
      l_lo = l_lo <= 0 ? 0 : l_lo / st;
      int l_hi = j / st;
      if (l_hi > L - 1) l_hi = L - 1;
      for (int l = l_lo; l <= l_hi; ++l) acc += proj[((long long)b * L + l) * pitch + (j - st * l)];
    }
    wav[i] = acc;
  }
}

int launch_decoder(const float* u, const float* Wd, int B, int L, int N, int K, int T, float* proj, float* wav,
                   cudaStream_t st) {
  VATSS_CHECK_ARG(K <= DEC_MAX_K, "decoder: kernel_size_enc %d > %d unsupported", K, DEC_MAX_K);
  const long long rows = (long long)B * L;
  if (rows == 0) return 0;
  k_decoder_proj<<<ceil_div(rows, 8), 256, (size_t)N * K * sizeof(float), st>>>(u, Wd, rows, N, K, proj);
  VATSS_LAUNCH_OK();
  return launch_decoder_ola(proj, K, B, L, K, T, wav, st);
}

// frames (B, L, pitch >= K) -> waveform (B, T): transposed-conv overlap-add with stride K/2 and the centred pad
int launch_decoder_ola(const float* proj, int pitch, int B, int L, int K, int T, float* wav, cudaStream_t st) {
  const int stride = K / 2;
  const int Lw = (L - 1) * stride + K;
  const int padl = (T - Lw) / 2;
  const long long total = (long long)B * T;
  int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  k_decoder_ola<<<blocks, 256, 0, st>>>(proj, pitch, L, K, stride, T, padl, total, wav);
  VATSS_LAUNCH_OK();
  return 0;
}

}  // namespace vatss
