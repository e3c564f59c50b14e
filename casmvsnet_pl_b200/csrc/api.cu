// C-ABI plumbing of libcasmvs.so: errors, device check, conv dispatch and the
// CostRegNet driver (models/mvsnet.py:60-104 of the reference).
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace casmvs {

std::atomic<uint64_t> g_launches{0};
std::atomic<uint64_t> g_fallbacks{0};
static thread_local char t_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_err, sizeof(t_err), fmt, ap);
  va_end(ap);
}

// conv3d_direct.cu
int conv3d_direct(const float* x, const float* wpk, const float* scale, const float* shift,
                  float slope, const float* skip, float* y, int B, int Cin, int Cout, int D,
                  int h, int w, int kind, int stride, cudaStream_t st, int round_out);
// conv3d_tma.cu (tcgen05 + TMA producer, persistent: the default stride-1 tensor path)
int conv3d_tma(const float* x, const float* wpk, const float* scale, const float* shift,
               float slope, const float* skip, float* y, int B, int Cin, int Cout, int D, int h,
               int w, int kind, int stride, int precision, cudaStream_t st);
// conv3d_tma_n8.cu (tcgen05 + TMA, stride-1 layers with Cout <= 8: kd and kw folded into N)
int conv3d_tma_n8(const float* x, const float* wpk, const float* scale, const float* shift,
                  float slope, const float* skip, float* y, int B, int Cin, int Cout, int D,
                  int h, int w, int kind, int stride, int precision, cudaStream_t st);
// conv3d_tma2.cu (tcgen05 + TMA producer, persistent: stride-2 and transposed layers)
int conv3d_tma2(const float* x, const float* wpk, const float* scale, const float* shift,
                float slope, const float* skip, float* y, int B, int Cin, int Cout, int D, int h,
                int w, int kind, int stride, int precision, cudaStream_t st);

struct LayerSpec { int cin, cout, kind, stride; };

// conv0..conv6, conv7, conv9, conv11, prob   (models/mvsnet.py:63-89)
static void costreg_layers(int Cin, LayerSpec (&L)[11]) {
  const LayerSpec t[11] = {
      {Cin, 8, CASMVS_CONV, 1},  {8, 16, CASMVS_CONV, 2},  {16, 16, CASMVS_CONV, 1},
      {16, 32, CASMVS_CONV, 2},  {32, 32, CASMVS_CONV, 1}, {32, 64, CASMVS_CONV, 2},
      {64, 64, CASMVS_CONV, 1},  {64, 32, CASMVS_CONV_TRANSPOSE, 2},
      {32, 16, CASMVS_CONV_TRANSPOSE, 2}, {16, 8, CASMVS_CONV_TRANSPOSE, 2},
      {8, 1, CASMVS_CONV, 1}};
  memcpy(L, t, sizeof(t));
}

}  // namespace casmvs

using namespace casmvs;

extern "C" int casmvs_version(void) { return CASMVS_VERSION; }
extern "C" const char* casmvs_last_error(void) { return t_err; }
extern "C" uint64_t casmvs_launch_count(void) { return g_launches.load(); }

extern "C" uint64_t casmvs_fallback_count(void) { return g_fallbacks.load(); }

extern "C" int casmvs_device_check(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    set_error("device_check: no CUDA device (%s)", cudaGetErrorString(e));
    return -3;
  }
  CASMVS_REQUIRE(device >= 0 && device < n, "device_check: device %d out of range (%d)", device, n);
  int major = 0, minor = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device);
  if (major != 10) {
    set_error("device_check: compute capability %d.%d; libcasmvs is built for sm_100a only "
              "(no fallback path)", major, minor);
    return -3;
  }
  return 0;
}

extern "C" int casmvs_conv3d_fwd(const float* x, const float* w_packed, const float* scale,
                                 const float* shift, float slope, const float* skip, float* y,
                                 int B, int Cin, int Cout, int D, int h, int w, int kind,
                                 int stride, int precision, void* stream) {
  CASMVS_REQUIRE(x && w_packed && y, "conv3d: null pointer");
  CASMVS_REQUIRE(B >= 0 && Cin > 0 && Cout > 0 && D > 0 && h > 0 && w > 0, "conv3d: bad dims");
  CASMVS_REQUIRE(Cin % 4 == 0, "conv3d: Cin must be a multiple of 4 (got %d)", Cin);
  CASMVS_REQUIRE(kind == CASMVS_CONV || kind == CASMVS_CONV_TRANSPOSE ||
                     kind == CASMVS_CONV_PLANAR, "conv3d: bad kind");
  CASMVS_REQUIRE(kind == CASMVS_CONV ? (stride == 1 || stride == 2)
                 : kind == CASMVS_CONV_PLANAR ? stride == 1 : stride == 2,
                 "conv3d: unsupported stride %d", stride);
  const int flags = precision & ~0xff;
  precision &= 0xff;
  CASMVS_REQUIRE((precision == CASMVS_FP32 || precision == CASMVS_TF32) &&
                     (flags & ~CASMVS_KEEP_FP32_OUT) == 0, "conv3d: bad precision %d", precision);
  if (B == 0) return 0;
  cudaStream_t st = as_stream(stream);
  if (precision == CASMVS_TF32) {
    const int pf = precision | flags;
    // tcgen05 kernels: each returns 0 (handled), <0 (failed) or 1 (shape not covered)
    int rc = conv3d_tma_n8(x, w_packed, scale, shift, slope, skip, y, B, Cin, Cout, D, h, w, kind,
                           stride, pf, st);
    if (rc <= 0) return rc;
    rc = conv3d_tma(x, w_packed, scale, shift, slope, skip, y, B, Cin, Cout, D, h, w, kind,
                    stride, pf, st);
    if (rc <= 0) return rc;
    if (kind != CASMVS_CONV_PLANAR) {
      rc = conv3d_tma2(x, w_packed, scale, shift, slope, skip, y, B, Cin, Cout, D, h, w, kind,
                       stride, pf, st);
      if (rc <= 0) return rc;
    }
    // no tensor-core kernel covers this layer shape: it runs on the CUDA cores (same TF32-rounded
    // storage convention).  Counted, so callers can assert the fast path was taken.
    g_fallbacks.fetch_add(1, std::memory_order_relaxed);
  }
  // in the tf32 modes every stored activation is tf32-rounded (unbiased operand for
  // the tensor-core layers); the prob head (Cout == 1) feeds the softmax and stays fp32
  const int round_out =
      (precision == CASMVS_TF32 && Cout > 1 && !(flags & CASMVS_KEEP_FP32_OUT)) ? 1 : 0;
  return conv3d_direct(x, w_packed, scale, shift, slope, skip, y, B, Cin, Cout, D, h, w, kind,
                       stride, st, round_out);
}

// ---- CostRegNet driver ------------------------------------------------------
// params blob: for each of the 11 layers in order, packed weights [27][cin][cout],
// then scale[cout], then shift[cout] (prob: scale = 1, shift = bias).
extern "C" size_t casmvs_costreg_param_floats(int Cin) {
  LayerSpec L[11];
  costreg_layers(Cin, L);
  size_t n = 0;
  for (auto& l : L) n += (size_t)27 * l.cin * l.cout + 2 * (size_t)l.cout;
  return n;
}

extern "C" int casmvs_costreg_layer_info(int Cin, int layer, int* cin, int* cout, int* kind,
                                         int* stride, size_t* w_off, size_t* scale_off,
                                         size_t* shift_off) {
  CASMVS_REQUIRE(layer >= 0 && layer < 11, "costreg_layer_info: layer %d out of range", layer);
  LayerSpec L[11];
  costreg_layers(Cin, L);
  size_t off = 0;
  for (int i = 0; i < layer; ++i) off += (size_t)27 * L[i].cin * L[i].cout + 2 * (size_t)L[i].cout;
  if (cin) *cin = L[layer].cin;
  if (cout) *cout = L[layer].cout;
  if (kind) *kind = L[layer].kind;
  if (stride) *stride = L[layer].stride;
  if (w_off) *w_off = off;
  off += (size_t)27 * L[layer].cin * L[layer].cout;
  if (scale_off) *scale_off = off;
  if (shift_off) *shift_off = off + L[layer].cout;
  return 0;
}

extern "C" size_t casmvs_costreg_workspace_bytes(int B, int Cin, int D, int h, int w) {
  (void)Cin;
  const size_t n = (size_t)B * D * h * w;
  // c0 8n | c1 2n | c2 2n | c3 n/2 | c4 n/2 | c5 n/8 | c6 n/8 | u7 n/2 | u9 2n | u11 8n
  return (8 * n + 2 * n + 2 * n + n / 2 + n / 2 + n / 8 + n / 8 + n / 2 + 2 * n + 8 * n + 64) *
         sizeof(float);
}

extern "C" int casmvs_costreg_fwd(const float* x, const float* params, float* logits, int B,
                                  int Cin, int D, int h, int w, int precision, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  CASMVS_REQUIRE(x && params && logits, "costreg: null pointer");
  CASMVS_REQUIRE(D % 8 == 0 && h % 8 == 0 && w % 8 == 0,
                 "costreg: D,h,w must be divisible by 8 (got %d,%d,%d)", D, h, w);
  const size_t need = casmvs_costreg_workspace_bytes(B, Cin, D, h, w);
  CASMVS_REQUIRE(workspace && workspace_bytes >= need, "costreg: workspace too small (%zu < %zu)",
                 workspace_bytes, need);
  if (B == 0) return 0;
  LayerSpec L[11];
  costreg_layers(Cin, L);
  const float *W[11], *SC[11], *SH[11];
  {
    size_t off = 0;
    for (int i = 0; i < 11; ++i) {
      W[i] = params + off; off += (size_t)27 * L[i].cin * L[i].cout;
      SC[i] = params + off; off += L[i].cout;
      SH[i] = params + off; off += L[i].cout;
    }
  }
  const size_t n = (size_t)B * D * h * w;
  float* ws = (float*)workspace;
  float* c0 = ws;            ws += 8 * n;
  float* c1 = ws;            ws += 2 * n;
  float* c2 = ws;            ws += 2 * n;
  float* c3 = ws;            ws += n / 2;
  float* c4 = ws;            ws += n / 2;
  float* c5 = ws;            ws += n / 8;
  float* c6 = ws;            ws += n / 8;
  float* u7 = ws;            ws += n / 2;
  float* u9 = ws;            ws += 2 * n;
  float* u11 = ws;
  const float slope = 0.01f;  // inplace_abn LeakyReLU default
  int rc;
#define LAYER(i, in, skip, out, d_, h_, w_, sl)                                                   \
  rc = casmvs_conv3d_fwd(in, W[i], SC[i], SH[i], sl, skip, out, B, L[i].cin, L[i].cout, d_, h_,  \
                         w_, L[i].kind, L[i].stride, precision, stream);                          \
  if (rc) return rc;
  LAYER(0, x, nullptr, c0, D, h, w, slope)
  LAYER(1, c0, nullptr, c1, D, h, w, slope)
  LAYER(2, c1, nullptr, c2, D / 2, h / 2, w / 2, slope)
  LAYER(3, c2, nullptr, c3, D / 2, h / 2, w / 2, slope)
  LAYER(4, c3, nullptr, c4, D / 4, h / 4, w / 4, slope)
  LAYER(5, c4, nullptr, c5, D / 4, h / 4, w / 4, slope)
  LAYER(6, c5, nullptr, c6, D / 8, h / 8, w / 8, slope)
  LAYER(7, c6, c4, u7, D / 8, h / 8, w / 8, slope)     // conv4 + conv7(x)   mvsnet.py:97
  LAYER(8, u7, c2, u9, D / 4, h / 4, w / 4, slope)     // conv2 + conv9(x)   mvsnet.py:99
  LAYER(9, u9, c0, u11, D / 2, h / 2, w / 2, slope)    // conv0 + conv11(x)  mvsnet.py:101
  LAYER(10, u11, nullptr, logits, D, h, w, 1.0f)       // prob: bias, no norm/act  :103
#undef LAYER
  return 0;
}
