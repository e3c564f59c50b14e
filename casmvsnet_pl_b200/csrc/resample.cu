// Input pipeline, device side: bilinear resize of uint8 RGB images, bit-exact with
// PIL.Image.resize(size, Image.BILINEAR) -- the network input of the reference's DTU, Tanks and
// BlendedMVS data sets (datasets/dtu.py:159-162, tanks.py, blendedmvs.py:162-163).
//
// PIL resamples separably in integer arithmetic: per output pixel a short run of taps, each an
// int32 weight with 22 fractional bits (built on the host in float64 by io.pil_bilinear_coeffs,
// the kernel only does the integer work).  A pass is
//     acc = 2^21 + sum_j pixel[xmin + j] * k[j]       (int32)
//     out = clamp(acc >> 22, 0, 255)
// The horizontal pass runs first and is clipped to uint8; the vertical pass runs on that uint8
// intermediate.  A pass whose axis keeps its size is skipped (PIL does not run it either).
//
// A CTA owns a kTH x kTW output tile.  It computes the horizontal pass for the input rows its
// vertical taps read into shared memory (uint8, exactly PIL's intermediate), then runs the
// vertical pass from there.  Rows beyond the staged window (only reachable through tables whose
// xmin is not PIL's near-linear ramp) are recomputed from global memory with the same integer
// function, so every table gives PIL's result.  Taps outside the image are skipped: PIL's are
// zero there.  HBM-bound and tiny next to a forward pass; its job is to take the resize off
// the host.
#include "common.cuh"

namespace casmvs {

constexpr int kTW = 64, kTH = 16, kThreads = 256;
constexpr int kSmemBudget = 48 * 1024;       // no opt-in: the datasets need a few KB

struct ResizeTables {
  const int* xmin_x;
  const int* taps_x;
  int kx;                                    // 0: no horizontal pass (W == w)
  const int* xmin_y;
  const int* taps_y;
  int ky;                                    // 0: no vertical pass (H == h)
};

static __device__ __forceinline__ uint8_t clip8(int acc) {
  const int v = acc >> 22;
  return (uint8_t)(v < 0 ? 0 : v > 255 ? 255 : v);
}

// horizontal pass of one input row at tile column xl -> 3 channels
static __device__ __forceinline__ void hpass(const uint8_t* __restrict__ row, int W, int x, int xl,
                                             const int* sxmin, const int* staps, int kx, uint8_t* dst) {
  if (kx == 0) {
    dst[0] = row[x * 3 + 0];
    dst[1] = row[x * 3 + 1];
    dst[2] = row[x * 3 + 2];
    return;
  }
  int a0 = 1 << 21, a1 = 1 << 21, a2 = 1 << 21;
  const int xmin = sxmin[xl];
  const int* k = staps + xl * kx;
  for (int j = 0; j < kx; ++j) {
    const int c = xmin + j;
    if ((unsigned)c < (unsigned)W) {
      const uint8_t* p = row + c * 3;
      a0 += p[0] * k[j];
      a1 += p[1] * k[j];
      a2 += p[2] * k[j];
    }
  }
  dst[0] = clip8(a0);
  dst[1] = clip8(a1);
  dst[2] = clip8(a2);
}

__global__ void __launch_bounds__(kThreads)
resize_u8_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, int H, int W, int h,
                 int w, ResizeTables t, int row_cap) {
  extern __shared__ __align__(16) unsigned char smem[];
  int* sxmin = reinterpret_cast<int*>(smem);                 // [kTW]
  int* staps_x = sxmin + kTW;                                // [kTW * kx]
  int* symin = staps_x + kTW * t.kx;                         // [kTH]
  int* staps_y = symin + kTH;                                // [kTH * ky]
  uint8_t* rows = reinterpret_cast<uint8_t*>(staps_y + kTH * t.ky);   // [row_cap][kTW * 3]
  __shared__ int s_r0, s_r1;

  const int x0 = blockIdx.x * kTW, y0 = blockIdx.y * kTH;
  const int tw = min(kTW, w - x0), th = min(kTH, h - y0);
  const uint8_t* img = in + (size_t)blockIdx.z * H * W * 3;
  uint8_t* dst = out + (size_t)blockIdx.z * h * w * 3;

  for (int i = threadIdx.x; i < tw; i += kThreads) {
    if (t.kx) sxmin[i] = t.xmin_x[x0 + i];
    for (int j = 0; j < t.kx; ++j) staps_x[i * t.kx + j] = t.taps_x[(size_t)(x0 + i) * t.kx + j];
  }
  for (int i = threadIdx.x; i < th; i += kThreads) {
    if (t.ky) symin[i] = t.xmin_y[y0 + i];
    for (int j = 0; j < t.ky; ++j) staps_y[i * t.ky + j] = t.taps_y[(size_t)(y0 + i) * t.ky + j];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    // input rows [r0, r1) the tile's vertical taps read, clipped to the image
    int r0 = y0, r1 = y0 + th;
    if (t.ky) {
      r0 = symin[0];
      r1 = symin[0] + t.ky;
      for (int i = 1; i < th; ++i) {
        r0 = min(r0, symin[i]);
        r1 = max(r1, symin[i] + t.ky);
      }
      r0 = max(r0, 0);
      r1 = min(r1, H);
    }
    s_r0 = r0;
    s_r1 = max(r0, min(r1, r0 + row_cap));
  }
  __syncthreads();
  const int r0 = s_r0, nstaged = s_r1 - s_r0;

  // horizontal pass of the staged rows (PIL's uint8 intermediate)
  for (int i = threadIdx.x; i < nstaged * tw; i += kThreads) {
    const int r = i / tw, xl = i - r * tw;
    hpass(img + (size_t)(r0 + r) * W * 3, W, x0 + xl, xl, sxmin, staps_x, t.kx,
          rows + (r * kTW + xl) * 3);
  }
  __syncthreads();

  // vertical pass
  for (int i = threadIdx.x; i < th * tw; i += kThreads) {
    const int yl = i / tw, xl = i - yl * tw;
    uint8_t v[3];
    if (t.ky == 0) {
      const int r = y0 + yl - r0;
      if (r < nstaged) {
        const uint8_t* s = rows + (r * kTW + xl) * 3;
        v[0] = s[0]; v[1] = s[1]; v[2] = s[2];
      } else {
        hpass(img + (size_t)(y0 + yl) * W * 3, W, x0 + xl, xl, sxmin, staps_x, t.kx, v);
      }
    } else {
      int a0 = 1 << 21, a1 = 1 << 21, a2 = 1 << 21;
      const int ymin = symin[yl];
      const int* k = staps_y + yl * t.ky;
      for (int j = 0; j < t.ky; ++j) {
        const int y = ymin + j;
        if ((unsigned)y >= (unsigned)H) continue;
        const int r = y - r0;
        uint8_t s[3];
        if (r >= 0 && r < nstaged) {
          const uint8_t* p = rows + (r * kTW + xl) * 3;
          s[0] = p[0]; s[1] = p[1]; s[2] = p[2];
        } else {
          hpass(img + (size_t)y * W * 3, W, x0 + xl, xl, sxmin, staps_x, t.kx, s);
        }
        a0 += s[0] * k[j];
        a1 += s[1] * k[j];
        a2 += s[2] * k[j];
      }
      v[0] = clip8(a0); v[1] = clip8(a1); v[2] = clip8(a2);
    }
    uint8_t* o = dst + ((size_t)(y0 + yl) * w + x0 + xl) * 3;
    o[0] = v[0]; o[1] = v[1]; o[2] = v[2];
  }
}

}  // namespace casmvs

using namespace casmvs;

extern "C" int casmvs_resize_u8_fwd(const uint8_t* in, int N, int H, int W, uint8_t* out, int h,
                                    int w, const int* xmin_x, const int* taps_x, int kx,
                                    const int* xmin_y, const int* taps_y, int ky, void* stream) {
  CASMVS_REQUIRE(in && out, "resize_u8: null image pointer");
  CASMVS_REQUIRE(N >= 0 && N <= 65535 && H > 0 && W > 0 && h > 0 && w > 0, "resize_u8: bad dims");
  if (W == w) {
    kx = 0;                                  // PIL skips a pass whose axis keeps its size
  } else {
    CASMVS_REQUIRE(xmin_x && taps_x && kx > 0, "resize_u8: W %d -> %d needs horizontal taps", W, w);
  }
  if (H == h) {
    ky = 0;
  } else {
    CASMVS_REQUIRE(xmin_y && taps_y && ky > 0, "resize_u8: H %d -> %d needs vertical taps", H, h);
  }
  if (N == 0) return 0;
  CASMVS_REQUIRE(in != out, "resize_u8: in-place resize is not supported");
  const long table_bytes = ((kTW * (kx + 1L) + kTH * (ky + 1L)) * 4 + 15) / 16 * 16;
  const long row_bytes = kTW * 3;
  CASMVS_REQUIRE(kx <= kSmemBudget && ky <= kSmemBudget && table_bytes + row_bytes <= kSmemBudget,
                 "resize_u8: %d horizontal x %d vertical taps do not fit shared memory", kx, ky);
  // input rows of one tile's vertical window: PIL's xmin moves by at most H / h + 1 per output
  // row, so (kTH - 1) * H / h + ky + 2 rows cover a tile.  A window larger than the budget is
  // staged in part; the kernel recomputes the remaining rows (see top).
  long rows_needed = ky ? (long)(kTH - 1) * H / h + ky + 2 : kTH;
  if (rows_needed > H) rows_needed = H;
  const long rows_fit = (kSmemBudget - table_bytes) / row_bytes;
  const int row_cap = (int)(rows_needed < rows_fit ? rows_needed : rows_fit);
  const int smem = (int)(table_bytes + row_cap * row_bytes);
  const ResizeTables t{xmin_x, taps_x, kx, xmin_y, taps_y, ky};
  dim3 grd((unsigned)((w + kTW - 1) / kTW), (unsigned)((h + kTH - 1) / kTH), (unsigned)N);
  resize_u8_kernel<<<grd, kThreads, smem, as_stream(stream)>>>(in, out, H, W, h, w, t, row_cap);
  return after_launch("resize_u8");
}
