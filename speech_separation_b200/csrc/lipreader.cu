// Lipreader front end (SURVEY.md §8f rank 4): the video feature extractor that produces the (512, Tv) lip embeddings
// the DPTN-AV model consumes - `Lipreading(modality="video", backbone_type="resnet", extract_feats=True)`,
// reference src/lipreader/lipreading/model.py:252-273 (forward), :180-207 (frontend3D), models/resnet.py:31-145
// (BasicBlock / ResNet-18 trunk), called from make_embeddings.py:58-66 and profiler.py:17-22.
//
//   video (B, T, Hin, Win) --crop + affine (dataloaders.py:24-27)--> (B, 1, T, 88, 88)
//     Conv3d(1->64, 5x7x7, stride 1x2x2, pad 2x3x3) + BatchNorm3d (eval) + act        -> (F, 44, 44, 64)   F = B T
//     MaxPool3d(1x3x3, stride 1x2x2, pad 0x1x1)                                        -> (F, 22, 22, 64)
//     8 BasicBlocks: act(bn2(conv2(act(bn1(conv1 x)))) + shortcut(x)), widths 64/128/256/512, stride 2 from layer2 on,
//       shortcut = 1x1 stride-2 conv + BN where the shape changes                      -> (F, 3, 3, 512)
//     AdaptiveAvgPool2d(1)                                                             -> (B, T, 512)
//
// Layout: activations are PIXEL-MAJOR (frame, y, x, channel) - one row of channels per pixel, like the token-major
// rows of the separation path - so a convolution is a GEMM over (pixels) x (taps x input channels) whose A rows are
// plain channel vectors.  BatchNorm (running statistics) is folded into a per-channel scale / shift at pack time.
// This file holds the fp32 engine (register-tiled implicit GEMM on the FMA pipe, exact to ~1e-6 against the fp32
// reference) and the packing kernels; lipreader_tc.cu holds the tcgen05 engine for the 3x3 / 1x1 trunk convolutions.
#include "common.cuh"
#include "lipreader.cuh"
#include "tc_kernels.cuh"

namespace vatss {

// ------------------------------------------------------------------------------------------
// geometry / packed layout (host)
// ------------------------------------------------------------------------------------------
int lip_conv_table(LipConv* t) {
  // conv 0: the 3-D front end (taps = 5*7*7, Cin = 1); then per BasicBlock conv1, conv2, shortcut (Cout = 0: none)
  int n = 0;
  size_t off = 0;
  auto add = [&](int taps, int cin, int cout, int ks, int stride, int pad) {
    LipConv c;
    c.taps = taps; c.cin = cin; c.cout = cout; c.ks = ks; c.stride = stride; c.pad = pad;
    c.off_w = off;   off += (size_t)taps * cin * cout * sizeof(float);
    c.off_scale = off; off += (size_t)cout * sizeof(float);
    c.off_shift = off; off += (size_t)cout * sizeof(float);
    c.off_slope = off; off += (size_t)cout * sizeof(float);
    c.off_w16 = off;   // tensor engine: K-major fp16 (the front end as a 64 x 256 matrix, taps zero-padded to 256)
    off += (cin >= 64) ? (size_t)taps * cin * cout * sizeof(__half) : (size_t)LIP_FRONT_K * cout * sizeof(__half);
    off = (off + 255) & ~(size_t)255;
    if (t) t[n] = c;
    ++n;
  };
  add(5 * 7 * 7, 1, 64, 7, 2, 3);
  int inpl = 64;
  const int widths[4] = {64, 128, 256, 512};
  for (int l = 0; l < 4; ++l)
    for (int b = 0; b < 2; ++b) {
      const int pl = widths[l], stride = (l > 0 && b == 0) ? 2 : 1;
      add(9, inpl, pl, 3, stride, 1);
      add(9, pl, pl, 3, 1, 1);
      if (stride != 1 || inpl != pl) add(1, inpl, pl, 1, stride, 0);
      else {
        LipConv c = {};
        c.off_w = c.off_scale = c.off_shift = c.off_slope = c.off_w16 = off;
        if (t) t[n] = c;
        ++n;
      }
      inpl = pl;
    }
  if (t) t[n].off_w = off;   // sentinel: total bytes
  return n;
}

size_t lip_packed_bytes() {
  LipConv t[LIP_NCONV + 1];
  lip_conv_table(t);
  return t[LIP_NCONV].off_w;
}

// ------------------------------------------------------------------------------------------
// packing kernels
// ------------------------------------------------------------------------------------------
// W (cout, cin, taps) fp32 -> Wp[(tap * cin + ci) * cout + co] fp32 and, for the tensor engine,
// W16[(co * taps + tap) * cin + ci] fp16 (K-major rows of one output channel: tap-major, channel-minor)
__global__ void k_lip_pack_w(const float* __restrict__ W, int cout, int cin, int taps, float* __restrict__ Wp,
                             __half* __restrict__ W16) {
  const long long n = (long long)cout * cin * taps;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int tap = (int)(i % taps);
    const int ci = (int)((i / taps) % cin);
    const int co = (int)(i / ((long long)taps * cin));
    const float w = W[i];
    Wp[((long long)tap * cin + ci) * cout + co] = w;
    if (W16) W16[((long long)co * taps + tap) * cin + ci] = __float2half_rn(w);
  }
}
// front end for the tensor engine: W (64, 1, 5, 7, 7) -> W16[co * 256 + tap], taps 245..255 zero
__global__ void k_lip_pack_front16(const float* __restrict__ W, __half* __restrict__ W16) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 64 * LIP_FRONT_K) return;
  const int tap = i % LIP_FRONT_K, co = i / LIP_FRONT_K;
  W16[i] = __float2half_rn(tap < 245 ? W[co * 245 + tap] : 0.f);
}
// eval-mode BatchNorm as y = x * scale + shift (torch: (x - mean) / sqrt(var + eps) * weight + bias, eps = 1e-5)
__global__ void k_lip_fold_bn(const float* __restrict__ g, const float* __restrict__ b, const float* __restrict__ rm,
                              const float* __restrict__ rv, const float* __restrict__ slope_in, int cout,
                              float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ slope) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cout) return;
  const float s = g[c] / sqrtf(rv[c] + 1e-5f);
  scale[c] = s;
  shift[c] = b[c] - rm[c] * s;
  slope[c] = slope_in ? slope_in[c] : 0.f;
}

int lip_pack(const float* const* params, int n_params, int relu_type, void* packed, size_t packed_bytes,
             cudaStream_t st) {
  VATSS_CHECK_ARG(params && n_params == LIP_NCONV * LIP_PSLOTS, "lipreader: parameter table must have %d entries",
                  LIP_NCONV * LIP_PSLOTS);
  VATSS_CHECK_ARG(relu_type >= LIP_ACT_RELU && relu_type <= LIP_ACT_SWISH, "lipreader: relu_type %d", relu_type);
  VATSS_CHECK_ARG(packed && packed_bytes >= lip_packed_bytes(), "lipreader: packed buffer too small");
  LipConv t[LIP_NCONV + 1];
  lip_conv_table(t);
  char* base = (char*)packed;
  for (int i = 0; i < LIP_NCONV; ++i) {
    const LipConv& c = t[i];
    const float* const* p = params + i * LIP_PSLOTS;
    if (c.cout == 0) {
      VATSS_CHECK_ARG(p[0] == nullptr, "lipreader: conv slot %d has no shortcut convolution but a weight was given", i);
      continue;
    }
    VATSS_CHECK_ARG(p[0] && p[1] && p[2] && p[3] && p[4], "lipreader: conv slot %d: missing weight / BatchNorm tensor", i);
    const bool is_shortcut = (i > 0 && (i - 1) % 3 == 2);
    VATSS_CHECK_ARG(relu_type != LIP_ACT_PRELU || is_shortcut || p[5], "lipreader: conv slot %d: PReLU slopes missing", i);
    const long long n = (long long)c.taps * c.cin * c.cout;
    k_lip_pack_w<<<ceil_div(n, 256) > 1184 ? 1184 : ceil_div(n, 256), 256, 0, st>>>(
        p[0], c.cout, c.cin, c.taps, (float*)(base + c.off_w), c.cin >= 64 ? (__half*)(base + c.off_w16) : nullptr);
    VATSS_LAUNCH_OK();
    if (i == 0) {
      k_lip_pack_front16<<<ceil_div(64 * LIP_FRONT_K, 256), 256, 0, st>>>(p[0], (__half*)(base + c.off_w16));
      VATSS_LAUNCH_OK();
    }
    k_lip_fold_bn<<<ceil_div(c.cout, 128), 128, 0, st>>>(p[1], p[2], p[3], p[4],
                                                         (relu_type == LIP_ACT_PRELU && !is_shortcut) ? p[5] : nullptr,
                                                         c.cout, (float*)(base + c.off_scale),
                                                         (float*)(base + c.off_shift), (float*)(base + c.off_slope));
    VATSS_LAUNCH_OK();
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
// activation (model.py:171-177, resnet.py:41-52)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float lip_act(float v, int act, float slope) {
  if (act == LIP_ACT_RELU) return fmaxf(v, 0.f);
  if (act == LIP_ACT_PRELU) return v >= 0.f ? v : v * slope;
  if (act == LIP_ACT_SWISH) return v * (1.0f / (1.0f + expf(-v)));   // x * sigmoid(x), models/swish.py:10
  return v;
}

// ------------------------------------------------------------------------------------------
// front end: Conv3d(1 -> 64, 5x7x7, stride 1x2x2, pad 2x3x3) + BN + act, crop / normalisation folded into the load
// ------------------------------------------------------------------------------------------
// CTA = (frame, 4 output rows x W1 columns); the 5 x 13 x (Wc + 8) input patch and all 245 x 64 weights sit in shared
// memory; thread = (two adjacent output pixels, 32-channel half): 245 taps x 64 FMAs against broadcast weight reads.
constexpr int LF_ROWS = 4;
constexpr int LF_CO = 64, LF_KT = 5, LF_KS = 7, LF_TAPS = LF_KT * LF_KS * LF_KS;

struct LipFrontArgs {
  const float* vid;   // (B, T, Hin, Win)
  int B, T, Hin, Win, y0, x0, Hc, Wc, H1, W1;
  float pre_scale, pre_shift;
  const float* Wp;    // [245][64]
  const float* scale; const float* shift; const float* slope;
  int act;
  float* out;         // (frames, H1, W1, 64) of the chunk
  __half* out16;      // optional fp16 copy (tensor engine)
  int f0, nf;         // frame chunk
};

__global__ void __launch_bounds__(192) k_lip_front3d(const LipFrontArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int npairs = (a.W1 + 1) / 2;
  const int PW = 4 * npairs + 8, PH = 2 * LF_ROWS + 5;   // PW >= Wc + 6, rows are 16-byte aligned
  float* Ws = smem;                       // 245 * 64
  float* patch = smem + LF_TAPS * LF_CO;  // 5 * PH * PW
  const int row_tiles = (a.H1 + LF_ROWS - 1) / LF_ROWS;
  // persistent: the 63 KB of weights are read once per CTA; a CTA walks a contiguous run of (frame, row tile) items
  for (int i = threadIdx.x; i < LF_TAPS * LF_CO / 4; i += blockDim.x)
    reinterpret_cast<float4*>(Ws)[i] = __ldg(reinterpret_cast<const float4*>(a.Wp) + i);
  const int total = a.nf * row_tiles;
  const int per = (total + gridDim.x - 1) / gridDim.x;
  const int it0 = blockIdx.x * per, it1 = (it0 + per < total) ? it0 + per : total;
  // thread = (output row r, pixel pair j, 32-channel half h): 2 x 32 accumulators, so a broadcast weight read feeds
  // two FMAs and the three 16-byte patch reads of a (kt, ky) row feed all 7 x 2 taps
  const int nthr = LF_ROWS * npairs;
  const int h = threadIdx.x / nthr, p = threadIdx.x % nthr;
  const int r = p / npairs, j = p % npairs;
  const int npatch = LF_KT * PH * PW;
  for (int item = it0; item < it1; ++item) {
    const int f = a.f0 + item / row_tiles, oy0 = (item % row_tiles) * LF_ROWS;
    const int b = f / a.T, t = f % a.T;
    __syncthreads();   // the previous item's patch is no longer read
    for (int i0 = threadIdx.x; i0 < npatch; i0 += 8 * 192) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {   // eight independent global loads in flight per thread
        const int i = i0 + u * 192;
        const int px = i % PW, py = (i / PW) % PH, kt = i / (PW * PH);
        const int tt = t + kt - 2, iy = 2 * oy0 - 3 + py, ix = px - 3;
        v[u] = 0.f;   // zero padding lives in the normalised domain
        if (i < npatch && tt >= 0 && tt < a.T && iy >= 0 && iy < a.Hc && ix >= 0 && ix < a.Wc)
          v[u] = __ldg(a.vid + (((long long)b * a.T + tt) * a.Hin + a.y0 + iy) * a.Win + a.x0 + ix) * a.pre_scale + a.pre_shift;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (i0 + u * 192 < npatch) patch[i0 + u * 192] = v[u];
    }
    __syncthreads();
    const int oy = oy0 + r;
    if (h >= 2 || oy >= a.H1) continue;
    float acc0[32], acc1[32];
#pragma unroll
    for (int q = 0; q < 32; ++q) acc0[q] = acc1[q] = 0.f;
    for (int kt = 0; kt < LF_KT; ++kt)
      for (int ky = 0; ky < LF_KS; ++ky) {
        const float4* pr = reinterpret_cast<const float4*>(patch + (kt * PH + 2 * r + ky) * PW + 4 * j);
        const float4 q0 = pr[0], q1 = pr[1], q2 = pr[2];
        const float pv[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
        const float* wrow = Ws + ((kt * LF_KS + ky) * LF_KS) * LF_CO + h * 32;
#pragma unroll
        for (int kx = 0; kx < LF_KS; ++kx) {
          const float va = pv[kx], vb = pv[kx + 2];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 w = *reinterpret_cast<const float4*>(wrow + kx * LF_CO + 4 * q);
            acc0[4 * q] = fmaf(va, w.x, acc0[4 * q]);         acc1[4 * q] = fmaf(vb, w.x, acc1[4 * q]);
            acc0[4 * q + 1] = fmaf(va, w.y, acc0[4 * q + 1]); acc1[4 * q + 1] = fmaf(vb, w.y, acc1[4 * q + 1]);
            acc0[4 * q + 2] = fmaf(va, w.z, acc0[4 * q + 2]); acc1[4 * q + 2] = fmaf(vb, w.z, acc1[4 * q + 2]);
            acc0[4 * q + 3] = fmaf(va, w.w, acc0[4 * q + 3]); acc1[4 * q + 3] = fmaf(vb, w.w, acc1[4 * q + 3]);
          }
        }
      }
#pragma unroll
    for (int q = 0; q < 32; ++q) {
      const int c = h * 32 + q;
      const float sc = a.scale[c], sh = a.shift[c], sl = a.slope[c];
      acc0[q] = lip_act(fmaf(acc0[q], sc, sh), a.act, sl);
      acc1[q] = lip_act(fmaf(acc1[q], sc, sh), a.act, sl);
    }
    const long long o = ((((long long)(f - a.f0)) * a.H1 + oy) * a.W1 + 2 * j) * LF_CO + h * 32;
#pragma unroll
    for (int q = 0; q < 8; ++q)
      *reinterpret_cast<float4*>(a.out + o + 4 * q) = make_float4(acc0[4 * q], acc0[4 * q + 1], acc0[4 * q + 2], acc0[4 * q + 3]);
    if (2 * j + 1 < a.W1) {
#pragma unroll
      for (int q = 0; q < 8; ++q)
        *reinterpret_cast<float4*>(a.out + o + LF_CO + 4 * q) =
            make_float4(acc1[4 * q], acc1[4 * q + 1], acc1[4 * q + 2], acc1[4 * q + 3]);
    }
  }
}

// Tensor engine: the front-end convolution as a GEMM.  This kernel writes the fp16 im2col matrix
//   A[(frame, oy, ox), tap] = video'[t + kt - 2, 2 oy + ky - 3, 2 ox + kx - 3],  tap = (kt 7 + ky) 7 + kx  (< 245, rest 0)
// (256 columns = 512 bytes per output pixel) and the 1 x 1 "convolution" kernel of lipreader_tc.cu contracts it with the
// 64 x 256 weight matrix (4 K slabs) - BatchNorm, activation and the fp16 store are that kernel's epilogue.
// CTA = (frame, 4 output rows): patch in shared memory as above, then thread = (pixel, 16-byte chunk of 8 taps):
// the 32 lanes of a warp write the 512 contiguous bytes of one pixel.
__global__ void __launch_bounds__(256) k_lip_im2col_front(const LipFrontArgs a, __half* __restrict__ A16) {
  extern __shared__ __align__(16) float smem[];
  const int PW = a.Wc + 6, PH = 2 * LF_ROWS + 5;
  float* patch = smem;                                                  // 5 * PH * PW
  int* tapoff = reinterpret_cast<int*>(smem + LF_KT * PH * PW);         // 256 offsets (-1: zero column)
  const int row_tiles = (a.H1 + LF_ROWS - 1) / LF_ROWS;
  const int f = a.f0 + blockIdx.x / row_tiles, oy0 = (blockIdx.x % row_tiles) * LF_ROWS;
  const int b = f / a.T, t = f % a.T;
  {
    const int tap = threadIdx.x;   // 256 threads
    const int kx = tap % LF_KS, ky = (tap / LF_KS) % LF_KS, kt = tap / (LF_KS * LF_KS);
    tapoff[tap] = tap < LF_TAPS ? (kt * PH + ky) * PW + kx : -1;
  }
  const int npatch = LF_KT * PH * PW;
  for (int i0 = threadIdx.x; i0 < npatch; i0 += 8 * 256) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = i0 + u * 256;
      const int px = i % PW, py = (i / PW) % PH, kt = i / (PW * PH);
      const int tt = t + kt - 2, iy = 2 * oy0 - 3 + py, ix = px - 3;
      v[u] = 0.f;
      if (i < npatch && tt >= 0 && tt < a.T && iy >= 0 && iy < a.Hc && ix >= 0 && ix < a.Wc)
        v[u] = __ldg(a.vid + (((long long)b * a.T + tt) * a.Hin + a.y0 + iy) * a.Win + a.x0 + ix) * a.pre_scale + a.pre_shift;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (i0 + u * 256 < npatch) patch[i0 + u * 256] = v[u];
  }
  __syncthreads();
  const int rows = (a.H1 - oy0 < LF_ROWS) ? a.H1 - oy0 : LF_ROWS;
  // thread = (16-byte chunk c of 8 taps, pixels p = warp, warp + 8, ...): the chunk - and with it the eight patch offsets -
  // is the same for every pixel a thread writes, so the offsets live in registers (the loop was bound by its 16 shared-memory
  // loads per 16 bytes stored: 8 offsets + 8 values)
  const int c = threadIdx.x & 31;
  int off[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) off[q] = tapoff[8 * c + q];
  const int npix = rows * a.W1;
  for (int p = threadIdx.x >> 5; p < npix; p += 8) {
    const int r = p / a.W1, ox = p - r * a.W1;
    const float* pb = patch + (2 * r) * PW + 2 * ox;
    uint32_t pk[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int o0 = off[2 * q], o1 = off[2 * q + 1];
      const __half2 h = __floats2half2_rn(o0 >= 0 ? pb[o0] : 0.f, o1 >= 0 ? pb[o1] : 0.f);
      pk[q] = *reinterpret_cast<const uint32_t*>(&h);
    }
    const long long row = (((long long)(f - a.f0)) * a.H1 + oy0 + r) * a.W1 + ox;
    *reinterpret_cast<uint4*>(A16 + row * LIP_FRONT_K + 8 * c) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
  }
}

// MaxPool 3x3, stride 2, pad 1 over (F, H, W, C) -> (F, Ho, Wo, C); one thread per 8 channels of an output pixel.
// The window is clamped instead of tested: a clamped coordinate always names a pixel that is inside the window anyway
// (row -1 -> row 0, row H -> row H - 1), so the maximum is unchanged, the nine loads are unconditional and all in flight.
struct LipV8 { float v[8]; };
__device__ __forceinline__ LipV8 lip_load8(const float* p) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  return LipV8{{a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}};
}
__device__ __forceinline__ LipV8 lip_load8(const __half* p) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
  const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&u.z)), d = __half22float2(*reinterpret_cast<const __half2*>(&u.w));
  return LipV8{{a.x, a.y, b.x, b.y, c.x, c.y, d.x, d.y}};
}
template <typename TIN>
__global__ void k_lip_maxpool(const TIN* __restrict__ in, int F, int H, int W, int C, int Ho, int Wo,
                              float* __restrict__ out, __half* __restrict__ out16) {
  const int c8 = C / 8;
  const long long n = (long long)F * Ho * Wo * c8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % c8);
    const int ox = (int)((i / c8) % Wo), oy = (int)((i / ((long long)c8 * Wo)) % Ho);
    const long long f = i / ((long long)c8 * Wo * Ho);
    LipV8 w[9];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      int iy = 2 * oy - 1 + ky;
      iy = iy < 0 ? 0 : (iy >= H ? H - 1 : iy);
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        int ix = 2 * ox - 1 + kx;
        ix = ix < 0 ? 0 : (ix >= W ? W - 1 : ix);
        w[ky * 3 + kx] = lip_load8(in + (((f * H + iy) * W + ix) * (long long)C) + 8 * c);
      }
    }
    float m[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      m[q] = w[0].v[q];
#pragma unroll
      for (int t = 1; t < 9; ++t) m[q] = fmaxf(m[q], w[t].v[q]);
    }
    const long long o = ((f * Ho + oy) * Wo + ox) * (long long)C + 8 * c;
    if (out) {
      *reinterpret_cast<float4*>(out + o) = make_float4(m[0], m[1], m[2], m[3]);
      *reinterpret_cast<float4*>(out + o + 4) = make_float4(m[4], m[5], m[6], m[7]);
    }
    if (out16) {
      const __half2 h0 = __floats2half2_rn(m[0], m[1]), h1 = __floats2half2_rn(m[2], m[3]);
      const __half2 h2 = __floats2half2_rn(m[4], m[5]), h3 = __floats2half2_rn(m[6], m[7]);
      *reinterpret_cast<uint4*>(out16 + o) = make_uint4(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1),
                                                         *reinterpret_cast<const uint32_t*>(&h2), *reinterpret_cast<const uint32_t*>(&h3));
    }
  }
}

// ------------------------------------------------------------------------------------------
// fp32 engine: 3x3 / 1x1 convolution as a register-tiled implicit GEMM
//   out[m, co] = act( (sum_{tap, ci} in[pix(m, tap), ci] * Wp[tap][ci][co]) * scale[co] + shift[co] + res[m, co] )
// ------------------------------------------------------------------------------------------
constexpr int LC_BM = 64, LC_BN = 64, LC_BK = 16;

struct LipConvArgs {
  const float* in;    // (F, H, W, Cin)
  int F, H, W, Cin, Ho, Wo, Cout, ks, stride, pad;
  const float* Wp; const float* scale; const float* shift; const float* slope;
  const float* res;   // (F, Ho, Wo, Cout) or NULL
  int act;
  float* out;
};

__global__ void __launch_bounds__(256) k_lip_conv_f32(const LipConvArgs a) {
  __shared__ __align__(16) float As[LC_BK][LC_BM + 4];
  __shared__ __align__(16) float Bs[LC_BK][LC_BN];
  const long long M = (long long)a.F * a.Ho * a.Wo;
  const long long m0 = (long long)blockIdx.x * LC_BM;
  const int n0 = blockIdx.y * LC_BN;
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  // loader roles: A - thread (row = tid / 4, 4 channels at (tid % 4) * 4); B - thread (k = tid / 16, 4 couts at tx * 4)
  const int arow = tid / 4, aq = tid % 4;
  const long long am = m0 + arow;
  int af = 0, aoy = 0, aox = 0;
  const bool arow_ok = am < M;
  if (arow_ok) {
    aox = (int)(am % a.Wo);
    aoy = (int)((am / a.Wo) % a.Ho);
    af = (int)(am / ((long long)a.Wo * a.Ho));
  }
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const int taps = a.ks * a.ks;
  for (int tap = 0; tap < taps; ++tap) {
    const int ky = tap / a.ks, kx = tap % a.ks;
    const int iy = aoy * a.stride + ky - a.pad, ix = aox * a.stride + kx - a.pad;
    const bool ok = arow_ok && iy >= 0 && iy < a.H && ix >= 0 && ix < a.W;
    const float* src = a.in + (((long long)af * a.H + iy) * a.W + ix) * a.Cin + aq * 4;
    const float* wsrc = a.Wp + ((long long)tap * a.Cin + ty) * a.Cout + n0 + tx * 4;
    for (int c0 = 0; c0 < a.Cin; c0 += LC_BK) {
      float4 av = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ok) av = *reinterpret_cast<const float4*>(src + c0);
      const float4 bv = *reinterpret_cast<const float4*>(wsrc + (long long)c0 * a.Cout);
      __syncthreads();
      As[aq * 4 + 0][arow] = av.x; As[aq * 4 + 1][arow] = av.y; As[aq * 4 + 2][arow] = av.z; As[aq * 4 + 3][arow] = av.w;
      *reinterpret_cast<float4*>(&Bs[ty][tx * 4]) = bv;
      __syncthreads();
#pragma unroll
      for (int k = 0; k < LC_BK; ++k) {
        const float4 x = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
        const float4 w = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
        const float xa[4] = {x.x, x.y, x.z, x.w}, wa[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(xa[i], wa[j], acc[i][j]);
      }
    }
  }
  const int c = n0 + tx * 4;
  const float4 sc = *reinterpret_cast<const float4*>(a.scale + c), sh = *reinterpret_cast<const float4*>(a.shift + c);
  const float4 sl = *reinterpret_cast<const float4*>(a.slope + c);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long m = m0 + ty * 4 + i;
    if (m >= M) continue;
    float4 v = make_float4(fmaf(acc[i][0], sc.x, sh.x), fmaf(acc[i][1], sc.y, sh.y), fmaf(acc[i][2], sc.z, sh.z),
                           fmaf(acc[i][3], sc.w, sh.w));
    if (a.res) {
      const float4 r = *reinterpret_cast<const float4*>(a.res + m * a.Cout + c);
      v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
    }
    v.x = lip_act(v.x, a.act, sl.x); v.y = lip_act(v.y, a.act, sl.y);
    v.z = lip_act(v.z, a.act, sl.z); v.w = lip_act(v.w, a.act, sl.w);
    *reinterpret_cast<float4*>(a.out + m * a.Cout + c) = v;
  }
}

// AdaptiveAvgPool2d(1): (F, HW, C) -> (F, C); fp32 or fp16 input
template <typename TIN>
__global__ void k_lip_avgpool(const TIN* __restrict__ in, int F, int HW, int C, float* __restrict__ out) {
  const long long n = (long long)F * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const long long f = i / C;
    float s = 0.f;
    for (int p = 0; p < HW; ++p) s += (float)in[(f * HW + p) * C + c];
    out[i] = s / (float)HW;
  }
}

// ------------------------------------------------------------------------------------------
// host: the launch sequence
// ------------------------------------------------------------------------------------------
static int out_dim(int n, int ks, int stride, int pad) { return (n + 2 * pad - ks) / stride + 1; }

int lip_geometry(int Hc, int Wc, LipGeom* g) {
  VATSS_CHECK_ARG(Hc >= 8 && Wc >= 8 && Wc <= 88 && Hc <= 1024, "lipreader: crop %d x %d unsupported (width <= 88)", Hc, Wc);
  g->H1 = out_dim(Hc, 7, 2, 3); g->W1 = out_dim(Wc, 7, 2, 3);
  g->H[0] = out_dim(g->H1, 3, 2, 1); g->W[0] = out_dim(g->W1, 3, 2, 1);
  for (int l = 1; l < 4; ++l) { g->H[l] = out_dim(g->H[l - 1], 3, 2, 1); g->W[l] = out_dim(g->W[l - 1], 3, 2, 1); }
  return 0;
}

// Per-frame pitch of each of the four trunk buffers: the largest trunk activation, max over layers of H_l W_l C_l.
// Layer 1 (H0 W0 64) for most crops, but layer 4 (H3 W3 512) for crops with a side of 8 - 12 pixels (8 x 8: 256 < 512).
static long long lip_trunk_frame_floats(const LipGeom& g) {
  long long m = 0;
  for (int l = 0; l < 4; ++l) {
    const long long v = (long long)g.H[l] * g.W[l] * (64 << l);
    m = v > m ? v : m;
  }
  return m;
}

static long long lip_frame_floats(const LipGeom& g) {
  // conv3d output + four trunk buffers
  return (long long)g.H1 * g.W1 * 64 + 4ll * lip_trunk_frame_floats(g);
}

int lip_chunk_frames(long long F) { return (int)(F < LIP_CHUNK ? F : LIP_CHUNK); }

void* g_lip_capture[LIP_NSTAGES] = {};

size_t lip_workspace_bytes(int B, int T, int Hc, int Wc) {
  LipGeom g;
  if (B <= 0 || T <= 0 || lip_geometry(Hc, Wc, &g)) return 0;
  const long long fc = lip_chunk_frames((long long)B * T);
  // fp32 buffers + fp16 shadows of the trunk buffers and the front end's im2col matrix (tensor engine) + slack
  return (size_t)(fc * lip_frame_floats(g) * 4 + fc * 4ll * lip_trunk_frame_floats(g) * 2 +
                  fc * (long long)g.H1 * g.W1 * LIP_FRONT_K * 2 + 4096);
}

int lip_forward(const void* packed, size_t packed_bytes, int relu_type, const float* video, int B, int T, int Hin,
                int Win, int y0, int x0, int Hc, int Wc, float pre_scale, float pre_shift, float* out, void* workspace,
                size_t workspace_bytes, int engine, cudaStream_t st) {
  VATSS_CHECK_ARG(packed && video && out && workspace, "lipreader: NULL pointer");
  VATSS_CHECK_ARG(packed_bytes >= lip_packed_bytes(), "lipreader: packed buffer too small");
  VATSS_CHECK_ARG(relu_type >= LIP_ACT_RELU && relu_type <= LIP_ACT_SWISH, "lipreader: relu_type %d", relu_type);
  VATSS_CHECK_ARG(B > 0 && T > 0 && y0 >= 0 && x0 >= 0 && y0 + Hc <= Hin && x0 + Wc <= Win,
                  "lipreader: crop (%d,%d)+(%d,%d) outside the %d x %d frame", y0, x0, Hc, Wc, Hin, Win);
  VATSS_CHECK_ARG(engine == VATSS_LIP_ENGINE_F32 || engine == VATSS_LIP_ENGINE_TENSOR, "lipreader: engine %d", engine);
  LipGeom g;
  if (int rc = lip_geometry(Hc, Wc, &g)) return rc;
  VATSS_CHECK_ARG(workspace_bytes >= lip_workspace_bytes(B, T, Hc, Wc), "lipreader: workspace too small");
  const int front_pairs = (g.W1 + 1) / 2;
  VATSS_CHECK_ARG(LF_ROWS * front_pairs * 2 <= 192, "lipreader: front-end tile does not fit (W1 = %d)", g.W1);
  LipConv t[LIP_NCONV + 1];
  lip_conv_table(t);
  const char* pk = (const char*)packed;
  const long long F = (long long)B * T;
  const int FC = lip_chunk_frames(F);
  float* buf0 = (float*)workspace;
  const long long trunk_floats = (long long)FC * lip_trunk_frame_floats(g);
  float* tb[4];
  for (int i = 0; i < 4; ++i) tb[i] = buf0 + (long long)FC * g.H1 * g.W1 * 64 + i * trunk_floats;
  __half* tb16[4];
  for (int i = 0; i < 4; ++i) tb16[i] = (__half*)(tb[3] + trunk_floats) + i * trunk_floats;
  __half* im2col16 = tb16[3] + trunk_floats;   // (FC, H1, W1, 256) fp16

  static PerDeviceOnce configured;
  const int front_smem = (LF_TAPS * LF_CO + LF_KT * (2 * LF_ROWS + 5) * (4 * front_pairs + 8)) * 4;
  if (configured.first())
    VATSS_CUDA_OK(cudaFuncSetAttribute(k_lip_front3d, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
  VATSS_CHECK_ARG(front_smem <= 100 * 1024, "lipreader: front-end patch too large");

  static PerDeviceOnce configured_im2col;
  const int im2col_smem = (LF_KT * (2 * LF_ROWS + 5) * (Wc + 6)) * 4 + 256 * 4;
  if (configured_im2col.first())
    VATSS_CUDA_OK(cudaFuncSetAttribute(k_lip_im2col_front, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
  VATSS_CHECK_ARG(im2col_smem <= 64 * 1024, "lipreader: front-end patch too large");

  for (long long f0 = 0; f0 < F; f0 += FC) {
    const int nf = (int)((F - f0) < FC ? (F - f0) : FC);
    const bool tc = engine == VATSS_LIP_ENGINE_TENSOR;
    // debug (vatss_debug_lipreader_capture): copy the stage just produced, (nf, per_frame) values, to its capture slot
    auto capture = [&](int slot, const void* src, long long per_frame) -> int {
      if (!g_lip_capture[slot]) return 0;
      const long long esz = tc ? (long long)sizeof(__half) : (long long)sizeof(float);
      VATSS_CUDA_OK(cudaMemcpyAsync((char*)g_lip_capture[slot] + f0 * per_frame * esz, src, nf * per_frame * esz,
                                    cudaMemcpyDeviceToDevice, st));
      return 0;
    };
    LipFrontArgs a;
    a.vid = video; a.B = B; a.T = T; a.Hin = Hin; a.Win = Win; a.y0 = y0; a.x0 = x0; a.Hc = Hc; a.Wc = Wc;
    a.H1 = g.H1; a.W1 = g.W1; a.pre_scale = pre_scale; a.pre_shift = pre_shift;
    a.Wp = (const float*)(pk + t[0].off_w); a.scale = (const float*)(pk + t[0].off_scale);
    a.shift = (const float*)(pk + t[0].off_shift); a.slope = (const float*)(pk + t[0].off_slope);
    a.act = relu_type; a.out = buf0; a.out16 = nullptr; a.f0 = (int)f0; a.nf = nf;
    const int items = nf * ((g.H1 + LF_ROWS - 1) / LF_ROWS);
    const long long npool = (long long)nf * g.H[0] * g.W[0] * 8;
    const int pool_grid = (int)(ceil_div(npool, 256) > 4736 ? 4736 : ceil_div(npool, 256));
    if (tc) {
      // im2col (fp16) -> GEMM with the 64 x 256 weight matrix on the tensor cores (+ BN + act) -> max pool
      k_lip_im2col_front<<<items, 256, im2col_smem, st>>>(a, im2col16);
      VATSS_LAUNCH_OK();
      LipConv cf = t[0];
      cf.taps = 1; cf.cin = LIP_FRONT_K; cf.ks = 1; cf.stride = 1; cf.pad = 0;
      __half* front16 = (__half*)buf0;   // (nf, H1, W1, 64) fp16 in the (unused) fp32 front-end buffer
      if (int rc = lip_conv_tc(pk, cf, im2col16, nf, g.H1, g.W1, g.H1, g.W1, nullptr, relu_type, front16, st)) return rc;
      if (int rc = capture(0, front16, (long long)g.H1 * g.W1 * 64)) return rc;
      k_lip_maxpool<__half><<<pool_grid, 256, 0, st>>>(front16, nf, g.H1, g.W1, 64, g.H[0], g.W[0], nullptr, tb16[0]);
      VATSS_LAUNCH_OK();
      if (int rc = capture(1, tb16[0], (long long)g.H[0] * g.W[0] * 64)) return rc;
    } else {
      const int slots = 2 * num_sms();
      k_lip_front3d<<<items < slots ? items : slots, 192, front_smem, st>>>(a);
      VATSS_LAUNCH_OK();
      if (int rc = capture(0, buf0, (long long)g.H1 * g.W1 * 64)) return rc;
      k_lip_maxpool<float><<<pool_grid, 256, 0, st>>>(buf0, nf, g.H1, g.W1, 64, g.H[0], g.W[0], tb[0], nullptr);
      VATSS_LAUNCH_OK();
      if (int rc = capture(1, tb[0], (long long)g.H[0] * g.W[0] * 64)) return rc;
    }
    int cur = 0, H = g.H[0], W = g.W[0], ci = 1, final_c = 64;
    for (int l = 0; l < 4; ++l)
      for (int b = 0; b < 2; ++b, ci += 3) {
        const LipConv &c1 = t[ci], &c2 = t[ci + 1], &cs = t[ci + 2];
        const int Ho = out_dim(H, 3, c1.stride, 1), Wo = out_dim(W, 3, c1.stride, 1);
        const int xb = cur, tbuf = (cur + 1) & 3, rb = (cur + 2) & 3, yb = (cur + 3) & 3;
        const int k = 2 * l + b;
        const long long out_frame = (long long)Ho * Wo * c1.cout;
        if (tc) {
          int rc = lip_conv_tc(pk, c1, tb16[xb], nf, H, W, Ho, Wo, nullptr, relu_type, tb16[tbuf], st);
          if (rc) return rc;
          if ((rc = capture(2 + 3 * k, tb16[tbuf], out_frame))) return rc;
          const __half* res = tb16[xb];
          if (cs.cout) {
            rc = lip_conv_tc(pk, cs, tb16[xb], nf, H, W, Ho, Wo, nullptr, LIP_ACT_NONE, tb16[rb], st);
            if (rc) return rc;
            if ((rc = capture(3 + 3 * k, tb16[rb], out_frame))) return rc;
            res = tb16[rb];
          }
          rc = lip_conv_tc(pk, c2, tb16[tbuf], nf, Ho, Wo, Ho, Wo, res, relu_type, tb16[yb], st);
          if (rc) return rc;
          if ((rc = capture(4 + 3 * k, tb16[yb], out_frame))) return rc;
        } else {
          auto run = [&](const LipConv& c, const float* in, int Hi, int Wi, const float* res, int act, float* o) -> int {
            LipConvArgs a;
            a.in = in; a.F = nf; a.H = Hi; a.W = Wi; a.Cin = c.cin; a.Ho = Ho; a.Wo = Wo; a.Cout = c.cout;
            a.ks = c.ks; a.stride = c.stride; a.pad = c.pad;
            a.Wp = (const float*)(pk + c.off_w); a.scale = (const float*)(pk + c.off_scale);
            a.shift = (const float*)(pk + c.off_shift); a.slope = (const float*)(pk + c.off_slope);
            a.res = res; a.act = act; a.out = o;
            dim3 grid(ceil_div((long long)nf * Ho * Wo, LC_BM), c.cout / LC_BN);
            k_lip_conv_f32<<<grid, 256, 0, st>>>(a);
            VATSS_LAUNCH_OK();
            return 0;
          };
          if (int rc = run(c1, tb[xb], H, W, nullptr, relu_type, tb[tbuf])) return rc;
          if (int rc = capture(2 + 3 * k, tb[tbuf], out_frame)) return rc;
          const float* res = tb[xb];
          if (cs.cout) {
            if (int rc = run(cs, tb[xb], H, W, nullptr, LIP_ACT_NONE, tb[rb])) return rc;
            if (int rc = capture(3 + 3 * k, tb[rb], out_frame)) return rc;
            res = tb[rb];
          }
          if (int rc = run(c2, tb[tbuf], Ho, Wo, res, relu_type, tb[yb])) return rc;
          if (int rc = capture(4 + 3 * k, tb[yb], out_frame)) return rc;
        }
        cur = yb; H = Ho; W = Wo; final_c = c2.cout;
      }
    const long long n = (long long)nf * final_c;
    if (tc) k_lip_avgpool<__half><<<ceil_div(n, 256), 256, 0, st>>>(tb16[cur], nf, H * W, final_c, out + f0 * final_c);
    else k_lip_avgpool<float><<<ceil_div(n, 256), 256, 0, st>>>(tb[cur], nf, H * W, final_c, out + f0 * final_c);
    VATSS_LAUNCH_OK();
  }
  return 0;
}

}  // namespace vatss
