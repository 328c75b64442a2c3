// C ABI of libvatss_b200.so (see include/vatss.h) and the host-side launch sequence of the
// forward pass.  No device allocation, no synchronisation, no throw across the boundary.
#include <stdarg.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"
#include "tensor_engine.cuh"
#include "tc_kernels.cuh"
#include "lipreader.cuh"

namespace vatss {

static thread_local std::string g_err;

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
}

// ---- instrumentation ---------------------------------------------------------------------
static std::atomic<unsigned long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

struct StageRecord { int stage; cudaEvent_t a, b; unsigned long long launches_at_begin, launches; };
static std::mutex g_prof_mu;
static std::atomic<bool> g_prof_on{false};   // read by stage_begin/end without the mutex
static std::vector<StageRecord> g_prof;
static int g_open[ST_COUNT];

void stage_begin(int stage, cudaStream_t st) {
  if (!g_prof_on) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  StageRecord r;
  r.stage = stage;
  if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
  cudaEventRecord(r.a, st);
  r.launches_at_begin = g_launches.load();
  r.launches = 0;
  g_open[stage] = (int)g_prof.size();
  g_prof.push_back(r);
}
void stage_end(int stage, cudaStream_t st) {
  if (!g_prof_on) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  const int i = g_open[stage];
  if (i < 0 || i >= (int)g_prof.size()) return;
  cudaEventRecord(g_prof[i].b, st);
  g_prof[i].launches = g_launches.load() - g_prof[i].launches_at_begin;
  g_open[stage] = -1;
}

static int stride_of(const vatss_model_desc* d) { return d->K / 2; }

static int check_desc(const vatss_model_desc* d) {
  VATSS_CHECK_ARG(d != nullptr, "model desc is NULL");
  VATSS_CHECK_ARG(d->kind >= VATSS_KIND_DPTN_AV && d->kind <= VATSS_KIND_DPRNN, "unknown model kind %d", d->kind);
  VATSS_CHECK_ARG(d->N > 0 && d->N % 4 == 0, "num_features=%d must be a positive multiple of 4", d->N);
  VATSS_CHECK_ARG(d->K >= 2, "kernel_size_enc=%d must be >= 2", d->K);
  VATSS_CHECK_ARG(d->H > 0 && d->num_blocks >= 0 && d->C > 0 && d->P > 0, "bad H/num_blocks/C/P");
  if (d->kind != VATSS_KIND_DPRNN)
    VATSS_CHECK_ARG(d->heads > 0 && d->N % d->heads == 0, "num_features=%d not divisible by heads=%d", d->N,
                    d->heads);
  if (d->kind == VATSS_KIND_DPTN_AV) VATSS_CHECK_ARG(d->E > 0, "video_emb_size must be > 0 for DPTN-AV");
  return 0;
}

static int n_params_of(const vatss_model_desc* d) {
  return VATSS_P_GLOBAL_COUNT + d->num_blocks * 2 * VATSS_S_COUNT;
}

static inline const float* sub_param(const float* const* params, int blk, int path, int slot) {
  return params[VATSS_P_GLOBAL_COUNT + (2 * blk + path) * VATSS_S_COUNT + slot];
}

// bump allocator over the caller's workspace (256-byte granules)
struct Bump {
  char* base;
  size_t off = 0;
  explicit Bump(void* p) : base(reinterpret_cast<char*>(p)) {}
  template <typename T>
  T* take(size_t count) {
    T* r = reinterpret_cast<T*>(base + off);
    off += ((count * sizeof(T) + 255) / 256) * 256;
    return r;
  }
};

struct Geometry {
  int B, T, Tv, L, S;
  long long tokens, frames;
};

static int geometry(const vatss_model_desc* d, int B, int T, int Tv, Geometry* g) {
  VATSS_CHECK_ARG(B > 0, "batch size %d must be positive", B);
  VATSS_CHECK_ARG(T >= d->K, "waveform length %d shorter than the encoder kernel %d", T, d->K);
  g->B = B; g->T = T; g->Tv = Tv;
  g->L = (T - d->K) / stride_of(d) + 1;
  VATSS_CHECK_ARG(g->L >= d->C, "encoded length %d shorter than one chunk (%d)", g->L, d->C);
  g->S = (g->L - d->C) / d->P + 1;
  g->tokens = (long long)B * g->S * d->C;
  g->frames = (long long)B * g->L;
  return 0;
}

struct GenericBuffers {
  float *enc, *vis, *xa, *xb, *qkv, *att, *tmp, *pre, *rnn, *y, *ola, *u, *hT, *hG, *proj;
};

static size_t carve_generic(const vatss_model_desc* d, const Geometry& g, void* ws, GenericBuffers* out) {
  Bump b(ws);
  const size_t N = d->N, H = d->H, tok = (size_t)g.tokens, fr = (size_t)g.frames;
  GenericBuffers r;
  r.enc = b.take<float>(fr * N);
  r.vis = b.take<float>(d->kind == VATSS_KIND_DPTN_AV ? (size_t)g.B * g.Tv * N : 0);
  r.xa = b.take<float>(tok * N);
  r.xb = b.take<float>(tok * N);
  r.qkv = b.take<float>(d->kind == VATSS_KIND_DPRNN ? 0 : tok * 3 * N);
  r.att = b.take<float>(d->kind == VATSS_KIND_DPRNN ? 0 : tok * N);
  r.tmp = b.take<float>(tok * N);
  r.pre = b.take<float>(tok * 8 * H);
  r.rnn = b.take<float>(tok * 2 * H);
  r.y = b.take<float>(tok * 2 * N);
  r.ola = b.take<float>(fr * 2 * N);
  r.u = b.take<float>(fr * N);
  r.hT = b.take<float>(d->kind == VATSS_KIND_DPTN_MASK ? fr * N : 0);
  r.hG = b.take<float>(d->kind == VATSS_KIND_DPTN_MASK ? fr * N : 0);
  r.proj = b.take<float>(fr * d->K);
  if (out) *out = r;
  return b.off;
}

static bool tensor_engine_selected(const vatss_model_desc* d) {
  if (d->engine == VATSS_ENGINE_GENERIC) return false;
  // DPRNN has no LayerNorm on its residual stream: rounding W_ih to fp16 alone costs 2-4e-3 of waveform error
  // (measured, DESIGN.md), above the 1e-3 tolerance.  The tensor engine therefore runs DPRNN with the hi/lo split
  // LSTM variant, which exists for N = 64 (the reference's dprnn.yaml); other widths stay on the GENERIC engine
  // unless the tensor engine is requested explicitly.
  if (d->kind == VATSS_KIND_DPRNN && d->N != 64 && d->engine != VATSS_ENGINE_TENSOR) return false;
  return tensor_engine_supports(d);
}

static int run_frontend(const vatss_model_desc* d, const float* const* params, const float* mix,
                        const float* emb1, const float* emb2, const Geometry& g, float* enc, float* seg,
                        __half* seg16, float* vis, cudaStream_t st) {
  const bool av = d->kind == VATSS_KIND_DPTN_AV;
  if (av) {
    VATSS_CHECK_ARG(emb1 && emb2 && g.Tv > 0, "DPTN-AV needs both lip-embedding streams (Tv=%d)", g.Tv);
    VATSS_CHECK_ARG(vis != nullptr, "DPTN-AV needs the visual scratch buffer");
    int rc = launch_visual_compress(emb1, emb2, params[VATSS_P_VIS_W], params[VATSS_P_VIS_B], g.B, d->E, g.Tv,
                                    d->N, vis, st);
    if (rc) return rc;
  }
  return launch_encoder(mix, params[VATSS_P_ENCODER_W], av ? vis : nullptr, params[VATSS_P_GATE],
                        params[VATSS_P_VLN_W], params[VATSS_P_VLN_B], g.B, g.T, g.Tv, d->N, d->K, g.L, g.S, d->C,
                        d->P, enc, seg, seg16, st);
}

// LSTM input projection for all directions: pre[:, dir*4H:(dir+1)*4H] = x Wih_dir^T + bih + bhh
static int generic_lstm(const vatss_model_desc* d, const float* const* params, int blk, int path,
                        const float* x, const SeqMap& map, int ndir, long long tokens, GenericBuffers& w,
                        cudaStream_t st) {
  const int H = d->H, N = d->N;
  {
  StageScope sc(ST_LSTM_INPUT, st);
  for (int dir = 0; dir < ndir; ++dir) {
    const int o = dir ? (VATSS_S_WIH_R - VATSS_S_WIH) : 0;
    int rc = launch_gemm_simt(x, N, sub_param(params, blk, path, VATSS_S_WIH + o),
                              sub_param(params, blk, path, VATSS_S_BIH + o),
                              sub_param(params, blk, path, VATSS_S_BHH + o), nullptr, 0, w.pre + dir * 4 * H,
                              (long long)ndir * 4 * H, tokens, 4 * H, N, 0, nullptr, st);
    if (rc) return rc;
  }
  }
  StageScope sc(ST_LSTM_RECURRENT, st);
  return launch_lstm_simt(w.pre, sub_param(params, blk, path, VATSS_S_WHH),
                          ndir == 2 ? sub_param(params, blk, path, VATSS_S_WHH_R) : nullptr, w.rnn, map, H, ndir,
                          st);
}

static int run_blocks_generic(const vatss_model_desc* d, const float* const* params, const Geometry& g,
                              GenericBuffers& w, cudaStream_t st) {
  const int N = d->N, H = d->H;
  const long long tok = g.tokens;
  int rc = 0;
  for (int blk = 0; blk < d->num_blocks; ++blk) {
    for (int path = 0; path < 2; ++path) {
      const SeqMap map = path == 0 ? intra_map(g.B, g.S, d->C) : inter_map(g.B, g.S, d->C);
      const int ndir = (path == 0 || d->bidir) ? 2 : 1;
      auto sp = [&](int slot) { return sub_param(params, blk, path, slot); };
      if (d->kind == VATSS_KIND_DPRNN) {
        // dprnn.py:37-45 / 78-87: LN(Linear(LSTM(z))) + z
        if ((rc = generic_lstm(d, params, blk, path, w.xa, map, ndir, tok, w, st))) return rc;
        {
          StageScope sc(ST_FFN_LN, st);
          if ((rc = launch_gemm_simt(w.rnn, ndir * H, sp(VATSS_S_FFN_W), sp(VATSS_S_FFN_B), nullptr, nullptr, 0,
                                     w.tmp, N, tok, N, ndir * H, 0, nullptr, st)))
            return rc;
          if ((rc = launch_layernorm(w.tmp, w.xa, sp(VATSS_S_LN2_W), sp(VATSS_S_LN2_B), w.xb, tok, N, 1, st)))
            return rc;
        }
        float* t = w.xa; w.xa = w.xb; w.xb = t;
      } else {
        // dptn.py:36-52
        {
          StageScope sc(ST_QKV, st);
          if ((rc = launch_gemm_simt(w.xa, N, sp(VATSS_S_INPROJ_W), sp(VATSS_S_INPROJ_B), nullptr, nullptr, 0,
                                     w.qkv, 3 * N, tok, 3 * N, N, 0, nullptr, st)))
            return rc;
        }
        {
          StageScope sc(ST_ATTENTION, st);
          if ((rc = launch_attention_simt(w.qkv, w.att, map, N, d->heads, st))) return rc;
        }
        {
          StageScope sc(ST_OUTPROJ_LN, st);
          if ((rc = launch_gemm_simt(w.att, N, sp(VATSS_S_OUTPROJ_W), sp(VATSS_S_OUTPROJ_B), nullptr, w.xa, N,
                                     w.tmp, N, tok, N, N, 0, nullptr, st)))
            return rc;
          if ((rc = launch_layernorm(w.tmp, nullptr, sp(VATSS_S_LN1_W), sp(VATSS_S_LN1_B), w.xb, tok, N, 0, st)))
            return rc;
        }
        if ((rc = generic_lstm(d, params, blk, path, w.xb, map, ndir, tok, w, st))) return rc;
        {
          StageScope sc(ST_FFN_LN, st);
          if ((rc = launch_gemm_simt(w.rnn, ndir * H, sp(VATSS_S_FFN_W), sp(VATSS_S_FFN_B), nullptr, w.xb, N,
                                     w.tmp, N, tok, N, ndir * H, 1, nullptr, st)))
            return rc;
          if ((rc = launch_layernorm(w.tmp, nullptr, sp(VATSS_S_LN2_W), sp(VATSS_S_LN2_B), w.xa, tok, N, 0, st)))
            return rc;
        }
      }
    }
  }
  return 0;
}

// PReLU -> speaker split -> overlap-add -> head -> decoder   (dptn_wav.py:47-59,186-194)
static int run_tail_generic(const vatss_model_desc* d, const float* const* params, const Geometry& g,
                            GenericBuffers& w, float* s1_pred, float* s2_pred, cudaStream_t st) {
  const int N = d->N;
  int rc;
  StageScope sc(ST_TAIL, st);
  if ((rc = launch_gemm_simt(w.xa, N, params[VATSS_P_SPK_W], params[VATSS_P_SPK_B], nullptr, nullptr, 0, w.y,
                             2 * N, g.tokens, 2 * N, N, 2, params[VATSS_P_PRELU], st)))
    return rc;
  if ((rc = launch_ola_token_major(w.y, g.B, g.S, d->C, d->P, g.L, 2 * N, w.ola, nullptr, st))) return rc;
  float* preds[2] = {s1_pred, s2_pred};
  for (int j = 0; j < 2; ++j) {
    if (d->kind == VATSS_KIND_DPTN_MASK) {
      if ((rc = launch_gemm_simt(w.ola + j * N, 2 * N, params[VATSS_P_HEAD_W], params[VATSS_P_HEAD_B], nullptr,
                                 nullptr, 0, w.hT, N, g.frames, N, N, 0, nullptr, st)))
        return rc;
      if ((rc = launch_gemm_simt(w.ola + j * N, 2 * N, params[VATSS_P_HGATE_W], params[VATSS_P_HGATE_B], nullptr,
                                 nullptr, 0, w.hG, N, g.frames, N, N, 0, nullptr, st)))
        return rc;
      if ((rc = launch_mask_combine(w.hT, w.hG, w.enc, w.u, g.frames * N, st))) return rc;
    } else {
      if ((rc = launch_gemm_simt(w.ola + j * N, 2 * N, params[VATSS_P_HEAD_W], params[VATSS_P_HEAD_B], nullptr,
                                 w.enc, N, w.u, N, g.frames, N, N, 0, nullptr, st)))
        return rc;
    }
    if ((rc = launch_decoder(w.u, params[VATSS_P_DECODER_W], g.B, g.L, N, d->K, g.T, w.proj, preds[j], st)))
      return rc;
  }
  return 0;
}

}  // namespace vatss

using namespace vatss;

extern "C" {

const char* vatss_last_error(void) { return g_err.c_str(); }
int vatss_abi_version(void) { return VATSS_ABI_VERSION; }

const char* vatss_engine_fallback_reason(const vatss_model_desc* d) {
  if (d == nullptr || d->engine == VATSS_ENGINE_GENERIC || tensor_engine_selected(d)) return nullptr;
  const char* why = tensor_engine_unsupported_reason(d);
  return why ? why : "DPRNN with num_features != 64 needs engine=\"tensor\" explicitly (precision, DESIGN.md 4)";
}

int vatss_frames(const vatss_model_desc* d, int T) {
  if (check_desc(d)) return -1;
  return T < d->K ? 0 : (T - d->K) / stride_of(d) + 1;
}
int vatss_chunks(const vatss_model_desc* d, int L) {
  if (check_desc(d)) return -1;
  return L < d->C ? 0 : (L - d->C) / d->P + 1;
}

size_t vatss_workspace_bytes(const vatss_model_desc* d, int B, int T, int Tv) {
  if (check_desc(d)) return 0;
  Geometry g;
  if (geometry(d, B, T, Tv, &g)) return 0;
  if (tensor_engine_selected(d)) return tensor_engine_workspace_bytes(d, g.B, g.T, g.Tv, g.L, g.S);
  return carve_generic(d, g, nullptr, nullptr);
}

size_t vatss_packed_weight_bytes(const vatss_model_desc* d) {
  if (check_desc(d)) return 0;
  if (!tensor_engine_selected(d)) return 0;
  return tensor_engine_packed_bytes(d);
}

int vatss_pack_weights(const vatss_model_desc* d, const float* const* params, int n_params, void* packed,
                       size_t packed_bytes, void* stream) {
  if (check_desc(d)) return -1;
  VATSS_CHECK_ARG(n_params == n_params_of(d), "parameter table has %d entries, expected %d", n_params,
                  n_params_of(d));
  if (!tensor_engine_selected(d)) return 0;
  VATSS_CHECK_ARG(packed != nullptr && packed_bytes >= tensor_engine_packed_bytes(d),
                  "packed weight buffer too small (%zu < %zu)", packed_bytes, tensor_engine_packed_bytes(d));
  return tensor_engine_pack(d, params, packed, (cudaStream_t)stream);
}

int vatss_forward(const vatss_model_desc* d, const float* const* params, int n_params, const void* packed,
                  const float* mix, const float* emb1, const float* emb2, int B, int T, int Tv, float* s1_pred,
                  float* s2_pred, void* workspace, size_t workspace_bytes, void* stream) {
  if (check_desc(d)) return -1;
  VATSS_CHECK_ARG(params != nullptr && n_params == n_params_of(d), "parameter table has %d entries, expected %d",
                  n_params, n_params_of(d));
  VATSS_CHECK_ARG(mix && s1_pred && s2_pred && workspace, "NULL tensor pointer passed to vatss_forward");
  Geometry g;
  if (geometry(d, B, T, Tv, &g)) return -1;
  const size_t need = vatss_workspace_bytes(d, B, T, Tv);
  VATSS_CHECK_ARG(workspace_bytes >= need, "workspace too small: %zu bytes given, %zu needed", workspace_bytes,
                  need);
  cudaStream_t st = (cudaStream_t)stream;
  if (tensor_engine_selected(d)) {
    VATSS_CHECK_ARG(packed != nullptr, "the tensor engine needs packed weights (call vatss_pack_weights)");
    return tensor_engine_forward(d, params, packed, mix, emb1, emb2, g.B, g.T, g.Tv, g.L, g.S, s1_pred, s2_pred,
                                 workspace, st);
  }
  GenericBuffers w;
  carve_generic(d, g, workspace, &w);
  int rc;
  {
    StageScope sc(ST_FRONTEND, st);
    if ((rc = run_frontend(d, params, mix, emb1, emb2, g, w.enc, w.xa, nullptr, w.vis, st))) return rc;
  }
  if ((rc = run_blocks_generic(d, params, g, w, st))) return rc;
  return run_tail_generic(d, params, g, w, s1_pred, s2_pred, st);
}

int vatss_segment(const float* x, int B, int N, int L, int C, int P, float* out, void* stream) {
  VATSS_CHECK_ARG(B >= 0 && N >= 0 && C > 0 && P > 0, "segment: bad shape");
  VATSS_CHECK_ARG(L >= C, "segment: length %d shorter than one chunk (%d)", L, C);
  if (B == 0 || N == 0) return 0;
  VATSS_CHECK_ARG(x && out, "segment: NULL pointer");
  return launch_segment_cm(x, B, N, L, C, P, out, (cudaStream_t)stream);
}

int vatss_overlap_add(const float* y, int B, int N, int S, int C, int P, float* out, void* stream) {
  VATSS_CHECK_ARG(B >= 0 && N >= 0 && S > 0 && C > 0 && P > 0, "overlap_add: bad shape");
  if (B == 0 || N == 0) return 0;
  VATSS_CHECK_ARG(y && out, "overlap_add: NULL pointer");
  return launch_overlap_add_cm(y, B, N, S, C, P, out, (cudaStream_t)stream);
}

int vatss_encoder(const vatss_model_desc* d, const float* const* params, const float* mix, const float* emb1,
                  const float* emb2, int B, int T, int Tv, float* enc_out, float* seg_out, float* vis_scratch,
                  void* stream) {
  if (check_desc(d)) return -1;
  VATSS_CHECK_ARG(params && mix && enc_out, "encoder: NULL pointer");
  Geometry g;
  if (geometry(d, B, T, Tv, &g)) return -1;
  return run_frontend(d, params, mix, emb1, emb2, g, enc_out, seg_out, nullptr, vis_scratch, (cudaStream_t)stream);
}

int vatss_decoder(const vatss_model_desc* d, const float* dec_w, const float* u, int B, int T, float* wav,
                  float* proj_scratch, void* stream) {
  if (check_desc(d)) return -1;
  VATSS_CHECK_ARG(dec_w && u && wav && proj_scratch, "decoder: NULL pointer");
  VATSS_CHECK_ARG(B > 0 && T >= d->K, "decoder: bad shape");
  const int L = (T - d->K) / stride_of(d) + 1;
  return launch_decoder(u, dec_w, B, L, d->N, d->K, T, proj_scratch, wav, (cudaStream_t)stream);
}

int vatss_tc_gemm(int epi, const void* A16, long long lda, const void* W16, const float* bias, const float* res,
                  long long ldr, const float* ln_w, const float* ln_b, float* out32, long long ldo32, void* out16,
                  long long ldo16, int act16, const float* prelu_a, long long M, int NOUT, int K, void* stream) {
  VATSS_CHECK_ARG(A16 && W16 && M >= 0, "tc_gemm: NULL operand");
  return launch_tc_gemm(epi, (const __half*)A16, lda, (const __half*)W16, bias, res, ldr, ln_w, ln_b, out32, ldo32,
                        (__half*)out16, ldo16, act16, prelu_a, M, NOUT, K, (cudaStream_t)stream);
}

int vatss_tc_gemm_ln16(const void* A16, long long lda, const void* W16, const float* bias, const void* res16,
                       long long ldr16, const float* ln_w, const float* ln_b, float* out32, long long ldo32,
                       void* out16, long long ldo16, int act16, const float* prelu_a, long long M, int NOUT, int K,
                       void* stream) {
  VATSS_CHECK_ARG(A16 && W16 && res16 && M >= 0, "tc_gemm_ln16: NULL operand");
  return launch_tc_gemm(TC_EPI_LN, (const __half*)A16, lda, (const __half*)W16, bias, nullptr, 0, ln_w, ln_b, out32,
                        ldo32, (__half*)out16, ldo16, act16, prelu_a, M, NOUT, K, (cudaStream_t)stream, nullptr, 0,
                        (const __half*)res16, ldr16);
}

int vatss_tc_lstm(const void* x16, const void* x16lo, const float* const* lp, void* out16, int mode, int B, int S, int C,
                  int N, int ndir, int act, void* wpack, float* bias_pack, void* stream) {
  VATSS_CHECK_ARG(x16 && lp && out16 && wpack && bias_pack, "tc_lstm: NULL pointer");
  VATSS_CHECK_ARG(ndir == 1 || ndir == 2, "tc_lstm: ndir must be 1 or 2");
  cudaStream_t st = (cudaStream_t)stream;
  for (int dir = 0; dir < ndir; ++dir) {
    int rc = launch_pack_lstm(lp[4 * dir + 0], lp[4 * dir + 1], lp[4 * dir + 2], lp[4 * dir + 3], N, dir,
                              x16lo != nullptr, (__half*)wpack, bias_pack, st);
    if (rc) return rc;
  }
  return launch_tc_lstm((const __half*)x16, (const __half*)x16lo, (const __half*)wpack, bias_pack, (__half*)out16, mode,
                        B, S, C, N, ndir,
                        act, st);
}

int vatss_tc_attention(const void* qkv16, void* out16, int mode, int B, int S, int C, int N, int heads, int force_simt,
                       void* stream) {
  VATSS_CHECK_ARG(qkv16 && out16 && heads > 0, "tc_attention: bad argument");
  const SeqMap map = mode == 0 ? intra_map(B, S, C) : inter_map(B, S, C);
  return launch_attention_f16((const __half*)qkv16, (__half*)out16, map, mode, B, S, C, N, heads, force_simt,
                              (cudaStream_t)stream);
}

int vatss_generic_gemm(const float* A, long long lda, const float* W, const float* bias, const float* bias2,
                       const float* R, long long ldr, float* out, long long ldc, long long M, int NOUT, int K, int act,
                       const float* prelu_a, void* stream) {
  VATSS_CHECK_ARG(A && W && out && M >= 0 && NOUT > 0 && K > 0, "generic_gemm: bad argument");
  VATSS_CHECK_ARG(act >= 0 && act <= 2 && (act != 2 || prelu_a), "generic_gemm: act %d needs its PReLU slope", act);
  return launch_gemm_simt(A, lda, W, bias, bias2, R, ldr, out, ldc, M, NOUT, K, act, prelu_a, (cudaStream_t)stream);
}

int vatss_generic_layernorm(const float* in, const float* res, const float* w, const float* b, float* out,
                            long long rows, int N, int mode, void* stream) {
  VATSS_CHECK_ARG(in && w && b && out && rows >= 0 && N > 0 && (mode == 0 || mode == 1),
                  "generic_layernorm: bad argument");
  return launch_layernorm(in, res, w, b, out, rows, N, mode, (cudaStream_t)stream);
}

int vatss_generic_attention(const float* qkv, float* out, int mode, int B, int S, int C, int N, int heads,
                            void* stream) {
  VATSS_CHECK_ARG(qkv && out && (mode == 0 || mode == 1) && B > 0 && S > 0 && C > 0 && N > 0,
                  "generic_attention: bad argument");
  const SeqMap map = mode == 0 ? intra_map(B, S, C) : inter_map(B, S, C);
  return launch_attention_simt(qkv, out, map, N, heads, (cudaStream_t)stream);
}

int vatss_generic_lstm(const float* pre, const float* whh_f, const float* whh_r, float* out, int mode, int B, int S,
                       int C, int H, int ndir, void* stream) {
  VATSS_CHECK_ARG(pre && whh_f && out && (ndir == 1 || (ndir == 2 && whh_r)), "generic_lstm: bad argument");
  VATSS_CHECK_ARG((mode == 0 || mode == 1) && B > 0 && S > 0 && C > 0, "generic_lstm: bad shape");
  const SeqMap map = mode == 0 ? intra_map(B, S, C) : inter_map(B, S, C);
  return launch_lstm_simt(pre, whh_f, whh_r, out, map, H, ndir, (cudaStream_t)stream);
}

int vatss_tc_tail(const vatss_model_desc* d, const float* const* params, int n_params, const void* packed,
                  const void* x16, const float* enc, int B, int T, float* s1_pred, float* s2_pred, void* workspace,
                  size_t workspace_bytes, void* stream) {
  if (check_desc(d)) return -1;
  VATSS_CHECK_ARG(params != nullptr && n_params == n_params_of(d), "parameter table has %d entries, expected %d",
                  n_params, n_params_of(d));
  VATSS_CHECK_ARG(tensor_engine_selected(d), "tc_tail: the model does not run on the TENSOR engine");
  VATSS_CHECK_ARG(packed && x16 && enc && s1_pred && s2_pred && workspace, "tc_tail: NULL pointer");
  Geometry g;
  if (geometry(d, B, T, 0, &g)) return -1;
  const size_t need = vatss_workspace_bytes(d, B, T, 0);
  VATSS_CHECK_ARG(workspace_bytes >= need, "workspace too small: %zu bytes given, %zu needed", workspace_bytes, need);
  return tensor_engine_tail(d, params, packed, (const __half*)x16, enc, g.B, g.T, 0, g.L, g.S, s1_pred, s2_pred,
                            workspace, (cudaStream_t)stream);
}

void vatss_debug_lstm_trace(void* dev_buffer) { vatss::g_lstm_trace = (long long*)dev_buffer; }
void vatss_debug_cta_limit(int ctas) { vatss::g_cta_limit = ctas; }
void vatss_debug_lstm_pingpong(int on) { vatss::g_lstm_pingpong = on; }
void vatss_debug_lstm_groups(int groups) { vatss::g_lstm_groups = groups; }
void vatss_debug_tail_staged(int on) { vatss::g_tail_staged = on; }
void vatss_debug_gemm_l2_order(int on) { vatss::g_gemm_l2_order = on; }
void vatss_debug_attention_version(int v) { vatss::g_attention_version = v == 1 ? 1 : 3; }

unsigned long long vatss_launch_count(void) { return g_launches.load(); }

int vatss_profile_begin(void) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (auto& r : g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  g_prof.clear();
  for (int i = 0; i < ST_COUNT; ++i) g_open[i] = -1;
  g_prof_on = true;
  return 0;
}

int vatss_profile_end(float* ms_per_stage, int* launches_per_stage, int n_stages) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_on = false;
  VATSS_CHECK_ARG(ms_per_stage && launches_per_stage && n_stages >= ST_COUNT, "profile_end: need %d slots", ST_COUNT);
  for (int i = 0; i < n_stages; ++i) { ms_per_stage[i] = 0.f; launches_per_stage[i] = 0; }
  int rc = 0;
  for (auto& r : g_prof) {
    float ms = 0.f;
    if (cudaEventSynchronize(r.b) != cudaSuccess || cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) rc = -2;
    ms_per_stage[r.stage] += ms;
    launches_per_stage[r.stage] += (int)r.launches;
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  g_prof.clear();
  if (rc) set_error("profile_end: event query failed");
  return rc;
}

int vatss_sisnr_chunks(int T) { return sisnr_chunks(T); }

int vatss_pit_sisnr(const float* s1p, const float* s2p, const float* s1, const float* s2, const float* mix, int B,
                    int T, double* rows_out, double* rows_loss_out, double* summary_out, double* scratch,
                    void* stream) {
  VATSS_CHECK_ARG(s1p && s2p && s1 && s2 && rows_out && rows_loss_out && summary_out && scratch,
                  "pit_sisnr: NULL pointer");
  StageScope sc(ST_SISNR, (cudaStream_t)stream);
  return launch_pit_sisnr(s1p, s2p, s1, s2, mix, B, T, rows_out, rows_loss_out, summary_out, scratch,
                          (cudaStream_t)stream);
}

int vatss_pit_sisnr_backward(const float* s1p, const float* s2p, const float* s1, const float* s2, int B, int T,
                             const double* scratch, const double* summary, const float* grad_out, float* grad_s1p,
                             float* grad_s2p, void* stream) {
  VATSS_CHECK_ARG(s1p && s2p && s1 && s2 && scratch && summary && grad_s1p && grad_s2p, "pit_sisnr_backward: NULL pointer");
  StageScope sc(ST_SISNR, (cudaStream_t)stream);
  return launch_pit_sisnr_backward(s1p, s2p, s1, s2, B, T, scratch, summary, grad_out, grad_s1p, grad_s2p,
                                   (cudaStream_t)stream);
}

int vatss_pit_sisdr(const float* s1p, const float* s2p, const float* s1, const float* s2, const float* mix, int B,
                    int T, int zero_mean, double* rows_out, double* summary_out, double* scratch, void* stream) {
  VATSS_CHECK_ARG(s1p && s2p && s1 && s2 && rows_out && summary_out && scratch, "pit_sisdr: NULL pointer");
  return launch_pit_sisdr(s1p, s2p, s1, s2, mix, B, T, zero_mean, rows_out, summary_out, scratch, (cudaStream_t)stream);
}

size_t vatss_sdr_workspace_bytes(int B, int T, int filter_length) { return sdr_workspace_bytes(B, T, filter_length); }

int vatss_sdr(const float* s1p, const float* s2p, const float* s1, const float* s2, const float* mix, int B, int T,
              int filter_length, int zero_mean, double load_diag, double* rows_out, double* summary_out,
              void* workspace, size_t workspace_bytes, void* stream) {
  VATSS_CHECK_ARG(s1p && s2p && s1 && s2 && rows_out && summary_out && workspace, "sdr: NULL pointer");
  return launch_sdr(s1p, s2p, s1, s2, mix, B, T, filter_length, zero_mean, load_diag, rows_out, summary_out, workspace,
                    workspace_bytes, (cudaStream_t)stream);
}

static int check_longform(int T, int W, int H) {
  VATSS_CHECK_ARG(T > 0 && W > 0, "longform: empty recording or window (T=%d, W=%d)", T, W);
  VATSS_CHECK_ARG(2 * (long long)H >= W && H < W, "longform: hop %d must satisfy W/2 <= hop < W (W=%d)", H, W);
  return 0;
}

int vatss_longform_windows(int T, int W, int H) {
  if (check_longform(T, W, H)) return -1;
  return longform_windows(T, W, H);
}

int vatss_window_cut(const float* mix, const float* emb1, const float* emb2, int R, int T, int Tv, int E, int W, int H,
                     int spf, int first, int count, float* mix_out, float* emb1_out, float* emb2_out, void* stream) {
  if (check_longform(T, W, H)) return -1;
  VATSS_CHECK_ARG(mix && mix_out, "window_cut: NULL pointer");
  VATSS_CHECK_ARG(R > 0 && R <= 65535, "window_cut: R=%d recordings out of range", R);
  const long long total = (long long)R * longform_windows(T, W, H);
  VATSS_CHECK_ARG(first >= 0 && count >= 0 && count <= 65535 && first + (long long)count <= total,
                  "window_cut: windows [%d, %d + %d) outside [0, %lld)", first, first, count, total);
  VATSS_CHECK_ARG((emb1 == nullptr) == (emb2 == nullptr) && (emb1 == nullptr) == (emb1_out == nullptr) &&
                      (emb1_out == nullptr) == (emb2_out == nullptr),
                  "window_cut: give both embeddings and both embedding outputs, or none");
  if (emb1) {
    VATSS_CHECK_ARG(E > 0 && Tv > 0, "window_cut: E=%d, Tv=%d must be positive", E, Tv);
    VATSS_CHECK_ARG(spf > 0 && W % spf == 0 && H % spf == 0,
                    "window_cut: window %d and hop %d must be multiples of samples_per_video_frame %d", W, H, spf);
  }
  return launch_window_cut(mix, emb1, emb2, R, T, Tv, E, W, H, spf, first, count, mix_out, emb1_out, emb2_out,
                           (cudaStream_t)stream);
}

size_t vatss_window_stitch_scratch_bytes(int R, int n) { return window_stitch_scratch_bytes(R, n); }

int vatss_window_stitch(const float* y1, const float* y2, int R, int T, int W, int H, float* s1, float* s2,
                        uint8_t* swaps_out, double* corr_out, void* scratch, size_t scratch_bytes, void* stream) {
  if (check_longform(T, W, H)) return -1;
  VATSS_CHECK_ARG(y1 && y2 && s1 && s2 && scratch, "window_stitch: NULL pointer");
  VATSS_CHECK_ARG(R > 0 && R <= 65535, "window_stitch: R=%d recordings out of range", R);
  const int n = longform_windows(T, W, H);
  VATSS_CHECK_ARG((long long)R * n < (1ll << 31), "window_stitch: %d x %d windows", R, n);
  const size_t need = window_stitch_scratch_bytes(R, n);
  VATSS_CHECK_ARG(scratch_bytes >= need, "window_stitch: scratch too small: %zu bytes given, %zu needed",
                  scratch_bytes, need);
  return launch_window_stitch(y1, y2, R, T, W, H, s1, s2, swaps_out, corr_out, scratch, (cudaStream_t)stream);
}

size_t vatss_stoi_workspace_bytes(int B, int T, int fs) { return stoi_workspace_bytes(B, T, fs); }

int vatss_stoi(const float* s1p, const float* s2p, const float* s1, const float* s2, int B, int T, int fs, int extended,
               double* rows_out, int* kept_out, double* summary_out, void* workspace, size_t workspace_bytes,
               void* stream) {
  VATSS_CHECK_ARG(s1p && s2p && s1 && s2 && rows_out && summary_out && workspace, "stoi: NULL pointer");
  return launch_stoi(s1p, s2p, s1, s2, B, T, fs, extended, rows_out, kept_out, summary_out, workspace,
                     workspace_bytes, (cudaStream_t)stream);
}

void vatss_debug_lipreader(int flags) { vatss::g_lip_dbg = flags; }
void vatss_debug_lipreader_kernel(int version) { vatss::g_lip_tc_version = version == 2 ? 2 : 1; }
void vatss_debug_lipreader_trace(void* dev_buffer) { vatss::g_lip_trace = (long long*)dev_buffer; }
void vatss_debug_lipreader_capture(void* const* stages, int n) {
  static_assert(vatss::LIP_NSTAGES == VATSS_LIP_NSTAGES, "stage count");
  for (int i = 0; i < vatss::LIP_NSTAGES; ++i) vatss::g_lip_capture[i] = (stages && i < n) ? stages[i] : nullptr;
}
size_t vatss_lipreader_packed_bytes(void) { return lip_packed_bytes(); }
size_t vatss_lipreader_workspace_bytes(int B, int T, int Hc, int Wc) { return lip_workspace_bytes(B, T, Hc, Wc); }
int vatss_lipreader_pack_weights(const float* const* params, int n_params, int relu_type, void* packed,
                                 size_t packed_bytes, void* stream) {
  return lip_pack(params, n_params, relu_type, packed, packed_bytes, (cudaStream_t)stream);
}
int vatss_lipreader_forward(const void* packed, size_t packed_bytes, int relu_type, const float* video, int B, int T,
                            int Hin, int Win, int y0, int x0, int Hc, int Wc, float pre_scale, float pre_shift,
                            float* out, void* workspace, size_t workspace_bytes, int engine, void* stream) {
  return lip_forward(packed, packed_bytes, relu_type, video, B, T, Hin, Win, y0, x0, Hc, Wc, pre_scale, pre_shift, out,
                     workspace, workspace_bytes, engine, (cudaStream_t)stream);
}

}  // extern "C"
