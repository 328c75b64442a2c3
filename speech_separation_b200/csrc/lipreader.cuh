// Lipreader front end: shared declarations of lipreader.cu (fp32 engine, packing, launch sequence) and
// lipreader_tc.cu (tcgen05 implicit-GEMM convolution).
#pragma once
#include "common.cuh"

namespace vatss {

enum { LIP_ACT_NONE = 0, LIP_ACT_RELU = 1, LIP_ACT_PRELU = 2, LIP_ACT_SWISH = 3 };
constexpr int LIP_NCONV = 25;    // front end + 8 blocks x (conv1, conv2, shortcut slot)
constexpr int LIP_PSLOTS = 6;    // per conv: weight, bn.weight, bn.bias, bn.running_mean, bn.running_var, prelu slopes
constexpr int LIP_FRONT_K = 256;  // front end on the tensor engine: 5 x 7 x 7 = 245 taps zero-padded to 4 K slabs
constexpr int LIP_CHUNK = 1024;  // frames per pass through the trunk (bounds the workspace)

struct LipConv {
  int taps, cin, cout, ks, stride, pad;
  size_t off_w, off_scale, off_shift, off_slope, off_w16;   // byte offsets into the packed buffer
};
struct LipGeom { int H1, W1, H[4], W[4]; };

int lip_conv_table(LipConv* t);   // fills t[0..LIP_NCONV], t[LIP_NCONV].off_w = total bytes
size_t lip_packed_bytes();
size_t lip_workspace_bytes(int B, int T, int Hc, int Wc);
int lip_geometry(int Hc, int Wc, LipGeom* g);
int lip_pack(const float* const* params, int n_params, int relu_type, void* packed, size_t packed_bytes, cudaStream_t st);
int lip_forward(const void* packed, size_t packed_bytes, int relu_type, const float* video, int B, int T, int Hin,
                int Win, int y0, int x0, int Hc, int Wc, float pre_scale, float pre_shift, float* out, void* workspace,
                size_t workspace_bytes, int engine, cudaStream_t st);

extern long long* g_lip_trace;
extern int g_lip_tc_version;
extern int g_lip_dbg;   // experiment switches of k_lip_conv_tc (0 in production)
constexpr int LIP_NSTAGES = 26;   // front end, pooled input, 8 blocks x (conv1, shortcut, output): VATSS_LIP_NSTAGES
extern void* g_lip_capture[LIP_NSTAGES];   // debug: per-stage copies of the next forwards (all NULL in production)

// tcgen05 engine: out16 (F, Ho, Wo, Cout) = act(conv(in16 (F, H, W, Cin)) * scale + shift + res16), fp16 activations,
// fp32 accumulation in TMEM
int lip_conv_tc(const char* packed, const LipConv& c, const __half* in16, int F, int H, int W, int Ho, int Wo,
                const __half* res16, int act, __half* out16, cudaStream_t st);

}  // namespace vatss
