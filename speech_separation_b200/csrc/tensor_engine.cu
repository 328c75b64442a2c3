// TENSOR engine: host-side launch sequence of the forward pass on the tcgen05 kernels.
//
// Residual stream: fp32 master copy + fp16 copy (the A operand of the next projection) written by the
// LayerNorm epilogues; every contraction runs on tcgen05 with fp16 operands and fp32 accumulation.
// (fp16 rather than bf16 operands: same tensor-core rate, and bf16 at every site misses the 1e-3
// waveform tolerance - SURVEY.md §7.3.)
#include "tensor_engine.cuh"

#include "tc_kernels.cuh"

#include <cstdlib>

namespace vatss {

// 1: the QKV and out-projection GEMMs walk their tiles in reverse, i.e. they start where their producers (FFN,
// attention) stopped and read the tail of x16 / att16 from L2 (VATSS_GEMM_L2_ORDER=0 / vatss_debug_gemm_l2_order(0):
// all kernels walk forwards).  Results do not depend on the order.
int g_gemm_l2_order = -1;
// 1: DPTN residual stream x as an fp16 hi / lo pair (no fp32 copy); 0: fp32 + fp16 copies (VATSS_X16SPLIT, experiments)
int g_x16split = -1;
static bool x16split_enabled() {
  if (g_x16split < 0) {
    const char* e = getenv("VATSS_X16SPLIT");
    g_x16split = e ? atoi(e) : 1;
  }
  return g_x16split != 0;
}

namespace {

inline const float* sub_param(const float* const* params, int blk, int path, int slot) {
  return params[VATSS_P_GLOBAL_COUNT + (2 * blk + path) * VATSS_S_COUNT + slot];
}

struct Bump {
  char* base;
  size_t off = 0;
  explicit Bump(void* p) : base(reinterpret_cast<char*>(p)) {}
  template <typename T>
  T* take(size_t count) {
    T* r = reinterpret_cast<T*>(base + off);
    off += ((count * sizeof(T) + 1023) / 1024) * 1024;
    return r;
  }
};

// ---- packed weights -----------------------------------------------------------------------
struct SubPacked {
  __half* win;     // [3N, N], q rows pre-scaled by log2(e)/sqrt(hd)
  float* bin;      // [3N]
  __half* wout;    // [N, N]
  __half* wffn;    // [N, ndir*H]
  __half* wlstm;   // [ndir][512][N+128]
  float* blstm;    // [ndir][512]
};
struct Packed {
  SubPacked sub[64];
  __half *wspk, *whead, *wgate;
  float *wfold, *wdT, *cfold;   // Wd^T Whead, Wd^T, Wd^T bhead (post-conv head folded into the decoder projection)
  float *w2, *c2;               // wfold Wspk[spk], wfold bspk[spk] (speaker split folded in as well)
};

size_t carve_packed(const vatss_model_desc* d, void* buf, Packed* out) {
  Bump b(buf);
  Packed p;
  const size_t N = d->N, H = d->H;
  const bool dprnn = d->kind == VATSS_KIND_DPRNN;
  for (int i = 0; i < d->num_blocks * 2; ++i) {
    const int ndir = (i % 2 == 0 || d->bidir) ? 2 : 1;
    SubPacked& s = p.sub[i];
    s.win = b.take<__half>(dprnn ? 0 : 3 * N * N);
    s.bin = b.take<float>(dprnn ? 0 : 3 * N);
    s.wout = b.take<__half>(dprnn ? 0 : N * N);
    s.wffn = b.take<__half>((dprnn ? 2 : 1) * N * ndir * H);   // DPRNN: [half(W) | half(W - half(W))]
    s.wlstm = b.take<__half>((size_t)ndir * 512 * ((dprnn ? 2 : 1) * N + 128));   // DPRNN: [W_hi | W_lo | W_hh]
    s.blstm = b.take<float>((size_t)ndir * 512);
  }
  p.wspk = b.take<__half>(2 * N * N);
  p.whead = b.take<__half>(N * N);
  p.wgate = b.take<__half>(d->kind == VATSS_KIND_DPTN_MASK ? N * N : 0);
  const bool fold = d->kind != VATSS_KIND_DPTN_MASK;   // post-conv head folded into the decoder projection
  p.wfold = b.take<float>(fold ? (size_t)d->K * N : 0);
  p.wdT = b.take<float>(fold ? (size_t)d->K * N : 0);
  p.cfold = b.take<float>(fold ? (size_t)d->K : 0);
  p.w2 = b.take<float>(fold ? (size_t)2 * d->K * N : 0);
  p.c2 = b.take<float>(fold ? (size_t)2 * d->K : 0);
  if (out) *out = p;
  return b.off;
}

// dst[i] = half(src[i] * (row < scaled_rows ? scale : 1))
__global__ void k_to_half(const float* __restrict__ src, __half* __restrict__ dst, long long n, int cols,
                          int scaled_rows, float scale) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float s = (i / cols) < scaled_rows ? scale : 1.f;
    dst[i] = __float2half_rn(src[i] * s);
  }
}
// dst[r, 0:cols] = half(src), dst[r, cols:2cols] = half(src - half(src))
__global__ void k_to_half_split(const float* __restrict__ src, __half* __restrict__ dst, int rows, int cols) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const int r = i / cols, c = i - r * cols;
  const float w = src[i];
  const __half hi = __float2half_rn(w);
  dst[(size_t)r * 2 * cols + c] = hi;
  dst[(size_t)r * 2 * cols + cols + c] = __float2half_rn(w - __half2float(hi));
}
__global__ void k_scale_bias(const float* __restrict__ src, float* __restrict__ dst, int n, int scaled, float scale) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i] * (i < scaled ? scale : 1.f);
}

int to_half(const float* src, __half* dst, long long rows, int cols, int scaled_rows, float scale, cudaStream_t st) {
  const long long n = rows * cols;
  k_to_half<<<(int)((n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184), 256, 0, st>>>(src, dst, n, cols, scaled_rows, scale);
  VATSS_LAUNCH_OK();
  return 0;
}

// ---- workspace ----------------------------------------------------------------------------
struct Work {
  float *enc32, *vis, *xa32, *xb32, *y32, *u32, *hT, *hG, *proj;
  __half *xa16, *xb16, *xa16lo, *xb16lo, *qkv16, *att16, *rnn16, *ola16;
};

size_t carve_work(const vatss_model_desc* d, int B, int Tv, int L, int S, void* buf, Work* out) {
  Bump b(buf);
  const size_t N = d->N, H = d->H, tok = (size_t)B * S * d->C, fr = (size_t)B * L;
  const bool dprnn = d->kind == VATSS_KIND_DPRNN, mask = d->kind == VATSS_KIND_DPTN_MASK;
  Work w;
  w.enc32 = b.take<float>(fr * N);
  w.vis = b.take<float>(d->kind == VATSS_KIND_DPTN_AV ? (size_t)B * Tv * N : 0);
  // fp32 residual stream: DPRNN keeps both ping-pong copies; the DPTN sub-blocks take the LayerNorm-1 output back as
  // fp16 (no xb32), and the fp16-stream variant drops the fp32 copy altogether
  const bool f16res = d->engine == VATSS_ENGINE_TENSOR_F16RES && !dprnn && !mask;
  // DPTN (not the masking model): the fp32 residual stream x is stored as the hi / lo fp16 pair (xa16, xa16lo) - xa16 is
  // the operand copy the projections read anyway, so x costs 4 bytes per element to write instead of 6
  const bool x16split = !dprnn && !mask && !f16res && x16split_enabled();
  w.xa32 = b.take<float>((f16res || x16split) ? 0 : tok * N);
  w.xb32 = b.take<float>(dprnn || mask ? tok * N : 0);   // (the masking head keeps y in fp32, see forward)
  w.xa16 = b.take<__half>(tok * N);
  w.xb16 = b.take<__half>(tok * N);
  w.xa16lo = b.take<__half>((dprnn || x16split) ? tok * N : 0);   // lo halves: hi/lo split LSTM input (DPRNN), residual x (DPTN)
  w.xb16lo = b.take<__half>(dprnn ? tok * N : 0);
  w.qkv16 = b.take<__half>(dprnn ? 0 : tok * 3 * N);
  w.att16 = b.take<__half>(dprnn ? 0 : tok * N);
  w.rnn16 = b.take<__half>(tok * 2 * H);
  // speaker-split output, overlap-add and head output exist only where the fused tail does not apply
  const bool unfused_tail = mask || !((N == 128 || N == 64) && (d->K == 7 || d->K == 2));
  w.y32 = b.take<float>(unfused_tail ? tok * 2 * N : 0);
  w.ola16 = b.take<__half>(unfused_tail ? fr * 2 * N : 0);
  w.u32 = b.take<float>(unfused_tail ? fr * N : 0);
  w.hT = b.take<float>(mask ? fr * N : 0);
  w.hG = b.take<float>(mask ? fr * N : 0);
  w.proj = b.take<float>(fr * 2 * d->K);
  if (out) *out = w;
  return b.off;
}

}  // namespace

// NULL when the tcgen05 kernels cover this model, else why they do not (reported once by the Python face: falling
// back to the fp32 SIMT engine is a ~20x performance cliff and must not be silent)
const char* tensor_engine_unsupported_reason(const vatss_model_desc* d) {
  if (d->H != 128) return "hidden_dim != 128 (the persistent LSTM kernel holds 512 x (N + 128) fp16 weights per CTA pair)";
  if (d->N != 128 && d->N != 64) return "num_features not in {64, 128}";
  if (d->kind == VATSS_KIND_DPRNN && d->N != 64) return "DPRNN: the hi/lo split LSTM exists for num_features = 64 only";
  if (d->kind != VATSS_KIND_DPRNN) {
    const int hd = d->N / d->heads;
    if (d->N % d->heads != 0 || (hd != 16 && hd != 32)) return "attention head dim not in {16, 32}";
  }
  if (d->num_blocks == 0) return "no dual-path blocks (the tail reads PReLU(x) from the last block's epilogue)";
  if (d->num_blocks > 32) return "more than 32 dual-path blocks";
  return nullptr;
}
bool tensor_engine_supports(const vatss_model_desc* d) { return tensor_engine_unsupported_reason(d) == nullptr; }

size_t tensor_engine_packed_bytes(const vatss_model_desc* d) { return carve_packed(d, nullptr, nullptr); }

size_t tensor_engine_workspace_bytes(const vatss_model_desc* d, int B, int T, int Tv, int L, int S) {
  (void)T;
  return carve_work(d, B, Tv, L, S, nullptr, nullptr);
}

int tensor_engine_pack(const vatss_model_desc* d, const float* const* params, void* packed, cudaStream_t st) {
  Packed p;
  carve_packed(d, packed, &p);
  const int N = d->N, H = d->H;
  const bool dprnn = d->kind == VATSS_KIND_DPRNN;
  int rc;
  if (g_gemm_l2_order < 0) {
    const char* e = getenv("VATSS_GEMM_L2_ORDER");
    g_gemm_l2_order = e ? atoi(e) : 1;
  }
  for (int blk = 0; blk < d->num_blocks; ++blk)
    for (int path = 0; path < 2; ++path) {
      const int ndir = (path == 0 || d->bidir) ? 2 : 1;
      SubPacked& s = p.sub[2 * blk + path];
      auto sp = [&](int slot) { return sub_param(params, blk, path, slot); };
      if (!dprnn) {
        const float qscale = 1.4426950408889634f / sqrtf((float)(N / d->heads));
        if ((rc = to_half(sp(VATSS_S_INPROJ_W), s.win, 3 * N, N, N, qscale, st))) return rc;
        k_scale_bias<<<(3 * N + 255) / 256, 256, 0, st>>>(sp(VATSS_S_INPROJ_B), s.bin, 3 * N, N, qscale);
        VATSS_LAUNCH_OK();
        if ((rc = to_half(sp(VATSS_S_OUTPROJ_W), s.wout, N, N, 0, 1.f, st))) return rc;
      }
      if (dprnn) {
        k_to_half_split<<<(N * ndir * H + 255) / 256, 256, 0, st>>>(sp(VATSS_S_FFN_W), s.wffn, N, ndir * H);
        VATSS_LAUNCH_OK();
      } else if ((rc = to_half(sp(VATSS_S_FFN_W), s.wffn, N, ndir * H, 0, 1.f, st))) return rc;
      for (int dir = 0; dir < ndir; ++dir) {
        const int o = dir ? (VATSS_S_WIH_R - VATSS_S_WIH) : 0;
        if ((rc = launch_pack_lstm(sp(VATSS_S_WIH + o), sp(VATSS_S_WHH + o), sp(VATSS_S_BIH + o), sp(VATSS_S_BHH + o),
                                   N, dir, dprnn ? 1 : 0, s.wlstm, s.blstm, st)))
          return rc;
      }
    }
  if ((rc = to_half(params[VATSS_P_SPK_W], p.wspk, 2 * N, N, 0, 1.f, st))) return rc;
  if ((rc = to_half(params[VATSS_P_HEAD_W], p.whead, N, N, 0, 1.f, st))) return rc;
  if (d->kind == VATSS_KIND_DPTN_MASK) {
    if ((rc = to_half(params[VATSS_P_HGATE_W], p.wgate, N, N, 0, 1.f, st))) return rc;
  } else if ((rc = launch_fold_head(params[VATSS_P_HEAD_W], params[VATSS_P_HEAD_B], params[VATSS_P_DECODER_W], N, d->K,
                                    p.wfold, p.wdT, p.cfold, st)) ||
             (rc = launch_fold_spk(p.wfold, params[VATSS_P_SPK_W], params[VATSS_P_SPK_B], N, d->K, p.w2, p.c2, st))) {
    return rc;
  }
  return 0;
}

int tensor_engine_forward(const vatss_model_desc* d, const float* const* params, const void* packed,
                          const float* mix, const float* emb1, const float* emb2, int B, int T, int Tv, int L,
                          int S, float* s1_pred, float* s2_pred, void* workspace, cudaStream_t st) {
  Packed p;
  carve_packed(d, const_cast<void*>(packed), &p);
  Work w;
  carve_work(d, B, Tv, L, S, workspace, &w);
  const int N = d->N, H = d->H, C = d->C;
  const long long tok = (long long)B * S * C;
  const bool dprnn = d->kind == VATSS_KIND_DPRNN, av = d->kind == VATSS_KIND_DPTN_AV;
  // DPTN residual stream.  Default: fp32 between sub-blocks, the LayerNorm-1 output y only as fp16 (it is the LSTM
  // operand anyway and re-enters as the FFN residual).  F16RES: the block residual is fp16 as well (1e-3 budget:
  // 3.8e-4 -> 5.7e-4 -> 7.0e-4 rel-L2 for fp32 / default / F16RES on the production goldens, DESIGN.md 4).
  const bool f16res = d->engine == VATSS_ENGINE_TENSOR_F16RES && !dprnn && d->kind != VATSS_KIND_DPTN_MASK;
  // the tanh x sigmoid masking head is the most sensitive consumer (7.2e-4 with the fp16 y, 9.1e-4 with the fp16
  // stream, 4.5e-4 without): it always keeps the fp32 residuals
  const bool y16res = d->kind != VATSS_KIND_DPTN_MASK;
  const bool x16split = !dprnn && d->kind != VATSS_KIND_DPTN_MASK && !f16res && x16split_enabled();   // x = xa16 + xa16lo (carve_work)
  int rc;
  {
    StageScope sc(ST_FRONTEND, st);
    if (av) {
      VATSS_CHECK_ARG(emb1 && emb2 && Tv > 0, "DPTN-AV needs both lip-embedding streams (Tv=%d)", Tv);
      if ((rc = launch_visual_compress(emb1, emb2, params[VATSS_P_VIS_W], params[VATSS_P_VIS_B], B, d->E, Tv, N, w.vis,
                                       st)))
        return rc;
    }
    if ((rc = launch_encoder(mix, params[VATSS_P_ENCODER_W], av ? w.vis : nullptr, params[VATSS_P_GATE],
                             params[VATSS_P_VLN_W], params[VATSS_P_VLN_B], B, T, Tv, N, d->K, L, S, C, d->P, w.enc32,
                             (f16res || x16split) ? nullptr : w.xa32, w.xa16, st, (dprnn || x16split) ? w.xa16lo : nullptr)))
      return rc;
  }
  for (int blk = 0; blk < d->num_blocks; ++blk)
    for (int path = 0; path < 2; ++path) {
      const int ndir = (path == 0 || d->bidir) ? 2 : 1;
      const SubPacked& s = p.sub[2 * blk + path];
      auto sp = [&](int slot) { return sub_param(params, blk, path, slot); };
      const SeqMap map = path == 0 ? intra_map(B, S, C) : inter_map(B, S, C);
      const bool last = (blk == d->num_blocks - 1) && path == 1;
      if (dprnn) {
        {
          StageScope sc(ST_LSTM_RECURRENT, st);
          if ((rc = launch_tc_lstm(w.xa16, w.xa16lo, s.wlstm, s.blstm, w.rnn16, path, B, S, C, N, ndir, 0, st))) return rc;
        }
        StageScope sc(ST_FFN_LN, st);
        if ((rc = launch_tc_gemm(TC_EPI_LN_POST, w.rnn16, ndir * H, s.wffn, sp(VATSS_S_FFN_B), w.xa32, N,
                                 sp(VATSS_S_LN2_W), sp(VATSS_S_LN2_B), w.xb32, N, w.xb16, N, last ? 2 : 0,
                                 params[VATSS_P_PRELU], tok, N, ndir * H, st, last ? nullptr : w.xb16lo, 1)))
          return rc;
        float* t32 = w.xa32; w.xa32 = w.xb32; w.xb32 = t32;
        __half* t16 = w.xa16; w.xa16 = w.xb16; w.xb16 = t16;
        t16 = w.xa16lo; w.xa16lo = w.xb16lo; w.xb16lo = t16;
      } else {
        {
          StageScope sc(ST_QKV, st);
          if ((rc = launch_tc_gemm(TC_EPI_F16, w.xa16, N, s.win, s.bin, nullptr, 0, nullptr, nullptr, nullptr, 0,
                                   w.qkv16, 3 * N, 0, nullptr, tok, 3 * N, N, st, nullptr, 0, nullptr, 0, g_gemm_l2_order)))
            return rc;
        }
        {
          StageScope sc(ST_ATTENTION, st);
          if ((rc = launch_attention_f16(w.qkv16, w.att16, map, path, B, S, C, N, d->heads, 0, st))) return rc;
        }
        {
          StageScope sc(ST_OUTPROJ_LN, st);
          if ((rc = launch_tc_gemm(TC_EPI_LN, w.att16, N, s.wout, sp(VATSS_S_OUTPROJ_B),
                                   (f16res || x16split) ? nullptr : w.xa32, N, sp(VATSS_S_LN1_W), sp(VATSS_S_LN1_B),
                                   y16res ? nullptr : w.xb32, N, w.xb16, N, 0, nullptr, tok, N, N, st, nullptr, 0,
                                   (f16res || x16split) ? w.xa16 : nullptr, N, g_gemm_l2_order,
                                   x16split ? w.xa16lo : nullptr)))
            return rc;
        }
        {
          StageScope sc(ST_LSTM_RECURRENT, st);
          if ((rc = launch_tc_lstm(w.xb16, nullptr, s.wlstm, s.blstm, w.rnn16, path, B, S, C, N, ndir, 1, st))) return rc;
        }
        StageScope sc(ST_FFN_LN, st);
        if ((rc = launch_tc_gemm(TC_EPI_LN, w.rnn16, ndir * H, s.wffn, sp(VATSS_S_FFN_B), y16res ? nullptr : w.xb32, N,
                                 sp(VATSS_S_LN2_W), sp(VATSS_S_LN2_B), (f16res || x16split || last) ? nullptr : w.xa32, N,
                                 w.xa16, N, last ? 2 : 0, params[VATSS_P_PRELU], tok, N, ndir * H, st,
                                 (x16split && !last) ? w.xa16lo : nullptr, 0, y16res ? w.xb16 : nullptr, N)))
          return rc;
      }
    }
  // the last block's epilogue left PReLU(x) in the fp16 copy
  return tensor_engine_tail(d, params, packed, w.xa16, w.enc32, B, T, Tv, L, S, s1_pred, s2_pred, workspace, st);
}

// tail: speaker split -> overlap-add -> head -> decoder, on x16 = PReLU(x) (fp16, token-major) and the encoder output
int tensor_engine_tail(const vatss_model_desc* d, const float* const* params, const void* packed, const __half* x16,
                       const float* enc32, int B, int T, int Tv, int L, int S, float* s1_pred, float* s2_pred,
                       void* workspace, cudaStream_t st) {
  Packed p;
  carve_packed(d, const_cast<void*>(packed), &p);
  Work w;
  carve_work(d, B, Tv, L, S, workspace, &w);
  const int N = d->N, C = d->C;
  const long long tok = (long long)B * S * C, fr = (long long)B * L;
  int rc;
  StageScope sc(ST_TAIL, st);
  float* preds[2] = {s1_pred, s2_pred};
  if (d->kind != VATSS_KIND_DPTN_MASK) {
    // speaker split + overlap-add + post-conv + skip + decoder projection: one gather over PReLU(x) (fp16) and enc
    rc = launch_tail_fused(x16, enc32, p.w2, p.c2, p.wdT, p.cfold, B, S, C, d->P, L, N, d->K, w.proj, st);
    if (rc < 0) return rc;
    if (rc == 0) {
      for (int j = 0; j < 2; ++j)
        if ((rc = launch_decoder_ola(w.proj + j * d->K, 2 * d->K, B, L, d->K, T, preds[j], st))) return rc;
      return 0;
    }
  }
  // no fused instance for (N, K), or the masking head: speaker split, overlap-add and head as separate passes
  if ((rc = launch_tc_gemm(TC_EPI_F32, x16, N, p.wspk, params[VATSS_P_SPK_B], nullptr, 0, nullptr, nullptr, w.y32,
                           2 * N, nullptr, 0, 0, nullptr, tok, 2 * N, N, st)))
    return rc;
  if ((rc = launch_ola_token_major(w.y32, B, S, C, d->P, L, 2 * N, nullptr, w.ola16, st))) return rc;
  for (int j = 0; j < 2; ++j) {
    if (d->kind == VATSS_KIND_DPTN_MASK) {
      if ((rc = launch_tc_gemm(TC_EPI_F32, w.ola16 + j * N, 2 * N, p.whead, params[VATSS_P_HEAD_B], nullptr, 0, nullptr,
                               nullptr, w.hT, N, nullptr, 0, 0, nullptr, fr, N, N, st)))
        return rc;
      if ((rc = launch_tc_gemm(TC_EPI_F32, w.ola16 + j * N, 2 * N, p.wgate, params[VATSS_P_HGATE_B], nullptr, 0, nullptr,
                               nullptr, w.hG, N, nullptr, 0, 0, nullptr, fr, N, N, st)))
        return rc;
      if ((rc = launch_mask_combine(w.hT, w.hG, enc32, w.u32, fr * N, st))) return rc;
    } else {
      if ((rc = launch_tc_gemm(TC_EPI_F32, w.ola16 + j * N, 2 * N, p.whead, params[VATSS_P_HEAD_B], enc32, N, nullptr,
                               nullptr, w.u32, N, nullptr, 0, 0, nullptr, fr, N, N, st)))
        return rc;
    }
    if ((rc = launch_decoder(w.u32, params[VATSS_P_DECODER_W], B, L, N, d->K, T, w.proj, preds[j], st))) return rc;
  }
  return 0;
}

}  // namespace vatss
