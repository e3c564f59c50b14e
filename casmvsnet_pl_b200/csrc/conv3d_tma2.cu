// K2 (tensor-core variant, TMA producer, part 2) — the stride-2 convolutions (conv1, conv3,
// conv5) and the transposed convolutions (conv7, conv9, conv11) of CostRegNet on tcgen05.
// The GEMMs ("resident brick + shifted-view UMMA descriptors", see conv3d_tma.cu):
//   MODE_S2 (stride 2): M = 8(w) x 16(h) OUTPUT voxels of one output slice od.  Input row
//     ih = 2*oh + kh - 1 => consecutive GEMM row groups are two brick rows apart; input column
//     iw = 2*ow + kw - 1 => even and odd columns are separate planes so that 8 consecutive ow are
//     again adjacent.  Odd input slices (s = 2a+1) feed outputs a (kd=2) and a+1 (kd=0) in ONE
//     MMA of N = 2*GW; even slices feed output a (kd=1).
//   MODE_T (transposed, output = 2x input): M = 8 x 16 INPUT voxels j of one input slice.
//     Output voxel o = 2j + p (p in {0,1}^3, 8 parity classes); class p reads input j + s with
//     tap k:  p=0 -> (s=0,k=1);  p=1 -> (s=0,k=2) and (s=1,k=0).  For each of the 4 in-plane
//     shifts (sh,sw) the A view is shared by every (class, kd) it reaches, so one MMA of
//     N = 12*Cout covers [kd=0 -> slice jd-1, pd=1 classes | kd=1 -> slice jd, pd=0 | kd=2 ->
//     slice jd, pd=1] with zero weight rows for unreachable classes (the MMA count, not N, is
//     what costs at these sizes: profiles/microbench/umma_rate.cu).
// How the input gets to shared memory and how the CTAs are scheduled:
//   * one or two TMA tiled loads per input slice (the first, cp.async generation of this kernel
//     issued 600-2400 16-byte copies per slice and was producer-bound);
//     out-of-bounds elements are zero-filled by the TMA unit (= the zero padding);
//   * the brick is voxel-major [rows][9 columns][CB channels], swizzled by its row size, and
//     every tap is a shifted view of it (start address + rows*9 + column, see conv3d_tma.cu);
//   * MODE_S2: the even and odd input columns are two planes, each loaded by a TMA whose box
//     walks W with element stride 2 (tensor map elementStrides = {1,2,1,1,1}); plane 0 holds
//     iw = 2*ow0-1+2j (taps kw = 0 at j, kw = 2 at j+1), plane 1 holds iw = 2*ow0+2j (kw = 1);
//     consecutive GEMM row groups are two brick rows apart (SBO = 2*9 voxels);
//   * persistent CTAs, 6 warps (0-3 epilogue, 4 TMA producer, 5 MMA issuer); accumulators are
//     re-zeroed by the epilogue after reading and handed back through tempty barriers.
//
//   * MODE_P5: the 5x5 stride-2 Conv2d layers of FeatureNet (conv1.0, conv2.0) as a planar
//     convolution over the (views, H, W) volume: the same even/odd planes (10 columns, 35 rows:
//     iw = 2*ow0-2+2j for kw = 0,2,4 at j, j+1, j+2; iw = 2*ow0-1+2j for kw = 1,3), 25 taps of
//     K = Cin, N = Cout, one accumulator group per image.
//
// Replaces (reference, relative to /root/reference):
//   ConvBnReLU(k=5, stride=2, pad=2)               models/modules.py:8-18, mvsnet.py:16,20
//   ConvBnReLU3D(stride=2)                         models/modules.py:21-31, mvsnet.py:65,68,71
//   ConvTranspose3d(k3,s2,p1,op1) + norm_act + skip models/mvsnet.py:74-87,99-101
#include <stdlib.h>

#include "common.cuh"
#include "tc_common.cuh"
#include "tma_common.cuh"

namespace casmvs {
namespace tma2 {

using namespace casmvs::tc;
using casmvs::tma::mbar_expect_tx;
using casmvs::tma::tma_load_5d;

enum { MODE_S2 = 0, MODE_T = 1, MODE_P5 = 2 };
constexpr int kThreads2 = 6 * 32;
constexpr int kProdWarp = 4, kIssueWarp = 5;

struct Params {
  const float* bimg;   // pre-built B operand image [chunk][tap][CIN/4][BROWS][4] (tf32-rounded)
  const float* scale;  // [Cout]
  const float* shift;  // [Cout]
  const float* skip;   // output-shaped or null
  float* y;            // (B,Do,Ho,Wo,Cout)
  float slope;
  int B, Di, Hi, Wi, Do, Ho, Wo, Cout;     // Cout = channel count of the output tensor;
                                           // a CTA handles the COUT-channel chunk blockIdx.y
  int tiles_w, tiles_h, nchunks, dchunk;   // tiles over the M space (output for S2, input for T)
  int round_out;
};

template <int MODE, int CIN, int COUT>
struct Cfg {
  static constexpr int CQ = CIN / 4;
  static constexpr int CB = CIN > 32 ? 32 : CIN;            // channels per brick plane
  static constexpr int NB = CIN / CB;
  static constexpr int ROWB = CB * 4;                       // bytes per voxel = swizzle span
  static constexpr int BR = MODE == MODE_S2 ? 33 : MODE == MODE_T ? 17 : 35;   // brick rows
  static constexpr int BW = MODE == MODE_P5 ? 10 : 9;       // brick columns per plane
  static constexpr int NPL = (MODE == MODE_T ? 1 : 2) * NB; // planes (= TMA loads) per slice
  static constexpr int kPlaneData = BR * BW * ROWB;
  static constexpr int kPlaneBytes = (kPlaneData + 1023) / 1024 * 1024;
  static constexpr int kSlotBytes = NPL * kPlaneBytes;
  // accumulator group (columns per output group) and B image rows per tap
  static constexpr int GW = MODE == MODE_T ? 8 * COUT : (COUT <= 16 ? 16 : 32);
  static constexpr int BROWS = MODE == MODE_S2 ? 3 * GW : MODE == MODE_T ? 12 * COUT : GW;
  static constexpr int NTAP = MODE == MODE_S2 ? 9 : MODE == MODE_T ? 4 : 25;   // A views per slice
  static constexpr int kWBytes = NTAP * CIN * BROWS * 4;
  static constexpr int kFixed = kWBytes + 2 * 32 * 4 + 192 + 32 * 8 + 32 * 8 + 1024;
  static constexpr int SLOTS = (kFixed + 4 * kSlotBytes <= 227 * 1024) ? 4
                               : (kFixed + 3 * kSlotBytes <= 227 * 1024) ? 3 : 2;
  static constexpr int kRingOff = 0;
  static constexpr int kWOff = SLOTS * kSlotBytes;
  static constexpr int kParamOff = kWOff + kWBytes;         // scale/shift [2][COUT pad 32]
  static constexpr int kBarOff = kParamOff + 2 * 32 * 4;
  // barriers: full[8] @0, empty[8] @64, tmem ptr @128, tfull[32] @192, tempty[32] @448
  static constexpr int kTotal = kBarOff + 192 + 32 * 8 + 32 * 8 + 1024;
  static constexpr uint32_t kLayout = ROWB == 128 ? 2u : ROWB == 64 ? 4u : 6u;
};

__host__ __device__ constexpr int tmem_cols_for2(int n) {
  return n <= 32 ? 32 : n <= 64 ? 64 : n <= 128 ? 128 : n <= 256 ? 256 : 512;
}

template <int MODE, int CIN, int COUT>
__global__ void __launch_bounds__(kThreads2, 1)
conv3d_tma2_kernel(const __grid_constant__ CUtensorMap xmap, const Params p) {
  using C = Cfg<MODE, CIN, COUT>;
  constexpr int BW = C::BW, GW = C::GW, BROWS = C::BROWS;
  constexpr int SLOTS = C::SLOTS;
  extern __shared__ unsigned char smem_raw[];
  const uint32_t s_raw = smem_u32(smem_raw);
  const uint32_t s_base = (s_raw + 1023u) & ~1023u;
  unsigned char* smem = smem_raw + (s_base - s_raw);
  const uint32_t s_ring = s_base + C::kRingOff, s_w = s_base + C::kWOff,
                 s_bar = s_base + C::kBarOff;
  float* s_param = reinterpret_cast<float*>(smem + C::kParamOff);
  const uint32_t bar_full = s_bar, bar_empty = s_bar + 64, bar_tfull = s_bar + 192,
                 bar_tempty = s_bar + 448, bar_w = s_bar + 136;   // bar_w: weight image landed
  volatile uint32_t* s_tmem_ptr = reinterpret_cast<volatile uint32_t*>(smem + C::kBarOff + 128);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t tmem_cols = tmem_cols_for2(p.dchunk * GW);
  const int total_items = p.B * p.nchunks * p.tiles_h * p.tiles_w;
  const int Dm = MODE == MODE_T ? p.Di : p.Do;               // M-space depth

  // ---- one-time setup ----
  {
    const int t = threadIdx.x;
    if (t < SLOTS) mbar_init(bar_full + 8 * t, 1);
    else if (t < 2 * SLOTS) mbar_init(bar_empty + 8 * (t - SLOTS), 1);
    else if (t >= 32 && t < 64) mbar_init(bar_tfull + 8 * (t - 32), 1);
    else if (t >= 64 && t < 96) mbar_init(bar_tempty + 8 * (t - 64), 128);
    else if (t == 96) mbar_init(bar_w, 1);
    if (t < 97) fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(smem_u32((const void*)s_tmem_ptr), tmem_cols);
  const int co_base = blockIdx.y * COUT;
  for (int i = threadIdx.x; i < 32; i += kThreads2) {
    s_param[i] = (i < COUT) ? (p.scale ? __ldg(p.scale + co_base + i) : 1.f) : 0.f;
    s_param[32 + i] = (i < COUT) ? (p.shift ? __ldg(p.shift + co_base + i) : 0.f) : 0.f;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem_ptr;
  if (threadIdx.x == 0) tma::load_image_bulk(s_w, p.bimg + (size_t)blockIdx.y * (C::kWBytes / 4), C::kWBytes, bar_w);
  if (warp < 4) {
    for (int c = 0; c < p.dchunk * GW; c += 16)
      tmem_zero16(tmem_base + ((uint32_t)(warp * 32) << 16) + c);
    tmem_wait_st();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  // nothing above depends on the previous kernel of the stream (see tma_common.cuh)
  tma::pdl_trigger();
  tma::pdl_wait();
  bool w_ready = false;                             // MMA issuer: weight image has landed
  uint32_t gs = 0;                                  // slices processed before this item
  int ep = 0;                                       // items processed by this CTA
  for (int item0 = blockIdx.x; item0 < total_items; item0 += gridDim.x, ++ep) {
    // ---- work item: (b, chunk of groups along depth, tile_h, tile_w) over the M space ----
    int item = item0;
    const int tw = item % p.tiles_w; item /= p.tiles_w;
    const int th = item % p.tiles_h; item /= p.tiles_h;
    const int ck = item % p.nchunks;
    const int b = item / p.nchunks;
    const int w0 = tw * kTileW, h0 = th * kTileH;            // M-space origin of the tile
    const int g0 = ck * p.dchunk, g1 = min(Dm, g0 + p.dchunk);
    const int ng = g1 - g0;                                  // accumulator groups of this item
    // input slices walked: S2: s = 2*g0-1 .. 2*g1-1  (2*ng+1);  T: s = g0 .. g1  (ng+1)
    // P5: s = g0 .. g1-1 (every image is its own group)
    const int nslices = MODE == MODE_S2 ? 2 * ng + 1 : MODE == MODE_T ? ng + 1 : ng;
    const int s_first = MODE == MODE_S2 ? 2 * g0 - 1 : g0;

    if (warp == kProdWarp) {
      // ===================== producer: NPL TMA loads per slice =====================
      if (lane == 0) {
        for (int it = 0; it < nslices; ++it) {
          const uint32_t g = gs + it;
          const int slot = g % SLOTS;
          if (g >= (uint32_t)SLOTS) mbar_wait(bar_empty + 8 * slot, ((g / SLOTS) - 1) & 1);
          const uint32_t dst = s_ring + slot * C::kSlotBytes;
          mbar_expect_tx(bar_full + 8 * slot, C::NPL * C::kPlaneData);
#pragma unroll
          for (int pl = 0; pl < C::NPL; ++pl) {
            const int nb = MODE == MODE_T ? pl : pl >> 1;
            const int wc = MODE == MODE_S2 ? 2 * w0 - 1 + (pl & 1)
                           : MODE == MODE_T ? w0 : 2 * w0 - 2 + (pl & 1);
            const int hc = MODE == MODE_S2 ? 2 * h0 - 1 : MODE == MODE_T ? h0 : 2 * h0 - 2;
            tma_load_5d(dst + pl * C::kPlaneBytes, &xmap, bar_full + 8 * slot, nb * C::CB, wc,
                        hc, s_first + it, b);
          }
        }
      }
      __syncwarp();
    } else if (warp == kIssueWarp) {
      // ===================== MMA issuer (warp-uniform, elect-predicated) =====================
      constexpr uint32_t a_lbo = 16;
      constexpr uint32_t a_sbo = (MODE == MODE_T ? 1 : 2) * BW * C::ROWB;
      constexpr uint32_t b_lbo = BROWS * 16, b_sbo = 128;
      constexpr int KPB = C::CB / 8;                          // K=8 steps per plane
      const uint32_t elected = elect_one();
      const uint64_t a_desc0 = make_desc(s_ring, a_lbo, a_sbo) | ((uint64_t)C::kLayout << 61);
      const uint64_t b_desc0 = make_desc(s_w, b_lbo, b_sbo);
      const uint32_t a_hi = (uint32_t)(a_desc0 >> 32), b_hi = (uint32_t)(b_desc0 >> 32);
      int waited = 0;                                         // groups handed back by the epilogue
      for (int it = 0; it < nslices; ++it) {
        const uint32_t g = gs + it;
        // which accumulator columns / B rows this input slice feeds
        int col, row0, ncols, done = -1, last;       // done: group completed by this slice
        if (MODE == MODE_S2) {
          if (it & 1) {                              // even input slice s = 2(g0+a): kd=1 -> group a
            const int a = (it - 1) >> 1;
            col = a * GW; row0 = 0; ncols = GW; last = a;
          } else {                                   // odd slice: kd=2 -> a-1, kd=0 -> a
            const int a = it >> 1;
            const int lo = max(a - 1, 0), hi = min(a, ng - 1);
            col = lo * GW;
            row0 = (a - 1 >= 0) ? GW : 2 * GW;       // rows [W1 | W2 | W0]
            ncols = (hi - lo + 1) * GW;
            if (a >= 1) done = a - 1;
            last = hi;
          }
        } else if (MODE == MODE_P5) {
          col = it * GW; row0 = 0; ncols = GW; done = it; last = it;
        } else {
          // T: slice it -> group it (blocks kd=1,kd=2; if it < ng) and group it-1 (block kd=0)
          const bool cur = it < ng, prev = it >= 1;
          col = prev ? (it - 1) * GW + 4 * COUT : 0;
          row0 = prev ? 0 : 4 * COUT;
          ncols = (prev ? 4 * COUT : 0) + (cur ? 8 * COUT : 0);
          if (prev) done = it - 1;
          last = cur ? it : it - 1;
        }
        const uint32_t idesc = make_idesc(128, ncols);
        const uint32_t acc = tmem_base + col;
        mbar_wait(bar_full + 8 * (g % SLOTS), (g / SLOTS) & 1);
        if (!w_ready) { mbar_wait(bar_w, 0); w_ready = true; }
        if (ep > 0) {
          for (; waited <= last; ++waited) mbar_wait(bar_tempty + 8 * waited, (ep - 1) & 1);
        }
        tc_fence_after();
        const uint32_t a_lo0 = (uint32_t)a_desc0 + (((g % SLOTS) * C::kSlotBytes) >> 4);
        const uint32_t b_lo0 = (uint32_t)b_desc0 + ((row0 * 16) >> 4);
#pragma unroll
        for (int tap = 0; tap < C::NTAP; ++tap) {
          int a_tap, pl0, plstep;                    // byte offset in a plane, first plane, planes per nb
          if (MODE == MODE_S2) {
            const int kh = tap / 3, kw = tap % 3;
            a_tap = (kh * BW + (kw == 2 ? 1 : 0)) * C::ROWB;
            pl0 = kw == 1 ? 1 : 0; plstep = 2;
          } else if (MODE == MODE_P5) {
            const int kh = tap / 5, kw = tap % 5;
            a_tap = (kh * BW + (kw >> 1)) * C::ROWB;
            pl0 = kw & 1; plstep = 2;
          } else {
            const int sh = tap >> 1, sw = tap & 1;
            a_tap = (sh * BW + sw) * C::ROWB;
            pl0 = 0; plstep = 1;
          }
#pragma unroll
          for (int k8 = 0; k8 < CIN / 8; ++k8) {
            const uint32_t a_off = ((pl0 + (k8 / KPB) * plstep) * C::kPlaneBytes + a_tap +
                                    (k8 % KPB) * 32) >> 4;
            const uint32_t b_off = (tap * (CIN * BROWS * 4) + k8 * 2 * BROWS * 16) >> 4;
            umma_tf32(acc, a_lo0 + a_off, a_hi, b_lo0 + b_off, b_hi, idesc, elected);
          }
        }
        if (done >= 0) umma_commit(bar_tfull + 8 * done, elected);
        umma_commit(bar_empty + 8 * (g % SLOTS), elected);
      }
      // groups a short chunk did not use still go through one empty -> full handshake per item
      for (int j = ng; j < p.dchunk; ++j) {
        if (ep > 0) {
          for (; waited <= j; ++waited) mbar_wait(bar_tempty + 8 * waited, (ep - 1) & 1);
        }
        if (elected) mbar_arrive(bar_tfull + 8 * j);
        __syncwarp();
      }
    } else {
      // ===================== epilogue warps 0..3 =====================
      const int m = warp * 32 + lane;
      const int mh = h0 + (m >> 3), mw = w0 + (m & 7);          // M-space voxel of this thread
      const uint32_t lane_base = tmem_base + ((uint32_t)(warp * 32) << 16);
      // MODE_T: the skip tensor (output-shaped, 8 parity classes per input voxel) is prefetched
      // in batches of 64 floats per thread BEFORE the accumulator is waited for, so its HBM
      // latency overlaps the MMAs instead of sitting in the epilogue's serial chain
      constexpr int CPB = COUT == 8 ? 8 : 4;                    // classes per skip batch
      constexpr int C4 = COUT / 4;
      float4 sk[MODE == MODE_T ? CPB * C4 : 1];
      auto load_skip = [&](int g, int cls0) {
        if constexpr (MODE == MODE_T) {
#pragma unroll
          for (int q = 0; q < CPB; ++q) {
            const int cc = cls0 + q;
            const int pd = cc >> 2, ph = (cc >> 1) & 1, pw = cc & 1;
            const int od = 2 * (g0 + g) + pd, oh = 2 * mh + ph, ow = 2 * mw + pw;
            const size_t o =
                ((((size_t)b * p.Do + od) * p.Ho + oh) * p.Wo + ow) * p.Cout + co_base;
#pragma unroll
            for (int c = 0; c < C4; ++c)
              sk[q * C4 + c] = (mh < p.Hi && mw < p.Wi) ? ldg4(p.skip + o + 4 * c)
                                                        : make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
      };
      for (int g = 0; g < p.dchunk; ++g) {
        if (MODE == MODE_T && p.skip && g < ng) load_skip(g, 0);
        mbar_wait(bar_tfull + 8 * g, ep & 1);
        if (g >= ng) {                                          // unused group: handshake only
          mbar_arrive(bar_tempty + 8 * g);
          continue;
        }
        tc_fence_after();
        if constexpr (MODE != MODE_T) {
          float acc[GW];
          tmem_ld<GW>(lane_base + g * GW, acc);
#pragma unroll
          for (int c = 0; c < GW; c += 16) tmem_zero16(lane_base + g * GW + c);
          tmem_wait_st();
          tc_fence_before();
          mbar_arrive(bar_tempty + 8 * g);                      // drained and zero again
          if (mh < p.Ho && mw < p.Wo) {
            const size_t o =
                ((((size_t)b * p.Do + (g0 + g)) * p.Ho + mh) * p.Wo + mw) * p.Cout + co_base;
#pragma unroll
            for (int c = 0; c < COUT; c += 4) {
              float v[4];
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                float t = fmaf(acc[c + k], s_param[c + k], s_param[32 + c + k]);
                t = t >= 0.f ? t : t * p.slope;
                v[k] = p.round_out ? to_tf32(t) : t;
              }
              st4(p.y + o + c, make_float4(v[0], v[1], v[2], v[3]));
            }
          }
        } else {
          // 8 classes x COUT columns: [pd][ph][pw][co]
#pragma unroll
          for (int cls = 0; cls < 8; ++cls) {
            constexpr int CW = COUT <= 16 ? 16 : 32;            // tcgen05.ld width
            float acc[CW];
            if constexpr (COUT == 8) {
              if (cls & 1) continue;                            // classes are read in pairs (16 cols)
              tmem_ld<16>(lane_base + g * GW + cls * COUT, acc);
              tmem_zero16(lane_base + g * GW + cls * COUT);
            } else {
              tmem_ld<CW>(lane_base + g * GW + cls * COUT, acc);
#pragma unroll
              for (int c = 0; c < CW; c += 16) tmem_zero16(lane_base + g * GW + cls * COUT + c);
            }
            if (cls == (COUT == 8 ? 6 : 7)) {                   // last read of the group
              tmem_wait_st();
              tc_fence_before();
              mbar_arrive(bar_tempty + 8 * g);
            }
            if (COUT != 8 && cls == CPB && p.skip) load_skip(g, CPB);   // second skip batch
            constexpr int NC = COUT == 8 ? 2 : 1;               // classes held in acc[]
#pragma unroll
            for (int q = 0; q < NC; ++q) {
              const int cc = cls + q;
              const int pd = cc >> 2, ph = (cc >> 1) & 1, pw = cc & 1;
              const int od = 2 * (g0 + g) + pd, oh = 2 * mh + ph, ow = 2 * mw + pw;
              if (mh < p.Hi && mw < p.Wi) {
                const size_t o =
                    ((((size_t)b * p.Do + od) * p.Ho + oh) * p.Wo + ow) * p.Cout + co_base;
#pragma unroll
                for (int c = 0; c < COUT; c += 4) {
                  float v[4];
#pragma unroll
                  for (int k = 0; k < 4; ++k) {
                    float t = fmaf(acc[q * COUT + c + k], s_param[c + k], s_param[32 + c + k]);
                    v[k] = t >= 0.f ? t : t * p.slope;
                  }
                  if (p.skip) {
                    const float4 s4 = sk[(cc % CPB) * C4 + c / 4];
                    v[0] += s4.x; v[1] += s4.y; v[2] += s4.z; v[3] += s4.w;
                  }
                  if (p.round_out) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) v[k] = to_tf32(v[k]);
                  }
                  st4(p.y + o + c, make_float4(v[0], v[1], v[2], v[3]));
                }
              }
            }
          }
        }
      }
    }
    gs += nslices;
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// B operand image [chunk][tap][cq][row][4], tf32-rounded
template <int MODE, int CIN, int COUT>
__global__ void build_image_tma2_kernel(const float* __restrict__ wpk, float* __restrict__ img,
                                        int cout_total) {
  using C = Cfg<MODE, CIN, COUT>;
  constexpr int CQ = C::CQ, GW = C::GW, BROWS = C::BROWS;
  constexpr int per = C::NTAP * CIN * BROWS;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < per * (cout_total / COUT);
       t += gridDim.x * blockDim.x) {
    const int ck = t / per, i = t - ck * per;
    const int jq = i & 3;
    const int row = (i >> 2) % BROWS;
    const int r = (i >> 2) / BROWS;          // tap*CQ + cq
    const int cq = r % CQ, tap = r / CQ;
    const int ci = cq * 4 + jq;
    int kd = -1, kh = -1, kw = -1, co = -1;
    if (MODE == MODE_S2) {
      // rows [W(kd=1) | W(kd=2) | W(kd=0)], tap = kh*3+kw
      const int g = row / GW;
      co = row % GW;
      kd = g == 0 ? 1 : g == 1 ? 2 : 0;
      kh = tap / 3; kw = tap % 3;
      if (co >= COUT) kd = -1;
    } else {
      // tap = sh*2+sw; rows: block 0 kd=0 (pd=1), block 1 kd=1 (pd=0), block 2 kd=2 (pd=1);
      // inside a block: class (ph,pw) = 2*ph+pw, then co
      const int sh = tap >> 1, sw = tap & 1;
      const int blk = row / (4 * COUT);
      const int cls = (row / COUT) & 3;
      co = row % COUT;
      const int ph = cls >> 1, pw = cls & 1;
      kd = blk;
      kh = sh == 0 ? (ph == 0 ? 1 : 2) : (ph == 1 ? 0 : -1);
      kw = sw == 0 ? (pw == 0 ? 1 : 2) : (pw == 1 ? 0 : -1);
      if (kh < 0 || kw < 0) kd = -1;
    }
    float v = 0.f;
    if (kd >= 0)
      v = to_tf32(__ldg(wpk + ((size_t)((kd * 3 + kh) * 3 + kw) * CIN + ci) * cout_total +
                        ck * COUT + co));
    img[t] = v;
  }
}

// MODE_P5 image [tap = kh*5+kw][cq][co (GW rows)][4] from the torch Conv2d weight (Cout,Cin,5,5)
template <int CIN, int COUT>
__global__ void build_image_p5_kernel(const float* __restrict__ wt, float* __restrict__ img) {
  using C = Cfg<MODE_P5, CIN, COUT>;
  constexpr int CQ = C::CQ, GW = C::GW;
  constexpr int total = 25 * CIN * GW;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
    const int jq = t & 3;
    const int co = (t >> 2) % GW;
    const int r = (t >> 2) / GW;             // tap*CQ + cq
    const int cq = r % CQ, tap = r / CQ;
    const int ci = cq * 4 + jq;
    img[t] = co < COUT ? to_tf32(__ldg(wt + ((size_t)co * CIN + ci) * 25 + tap)) : 0.f;
  }
}

template <int MODE, int CIN, int COUT>
static int launch2(const float* x, const float* wpk, Params p, cudaStream_t st) {
  using C = Cfg<MODE, CIN, COUT>;
  static_assert(C::kTotal <= 227 * 1024, "shared memory budget");
  auto kfn = conv3d_tma2_kernel<MODE, CIN, COUT>;
  static std::atomic<bool> attr_set[kMaxDevices];
  if (int rc = opt_in_smem(kfn, C::kTotal, attr_set, "conv3d_tma2")) return rc;
  // S2: box {CB, 17 traversed -> 9 loaded, 33, 1, 1} walking W with stride 2; T: {CB, 9, 17}
  // P5: box {CB, 19 traversed -> 10 loaded, 35, 1, 1} walking W with stride 2
  const CUtensorMap* map =
      MODE == MODE_S2   ? tma::input_map(x, p.B, p.Di, p.Hi, p.Wi, CIN, C::CB, 17, C::BR, 2)
      : MODE == MODE_P5 ? tma::input_map(x, p.B, p.Di, p.Hi, p.Wi, CIN, C::CB, 19, C::BR, 2)
                        : tma::input_map(x, p.B, p.Di, p.Hi, p.Wi, CIN, C::CB, C::BW, C::BR, 1);
  if (!map) return -2;
  static int per_sm_env = -1;
  if (per_sm_env < 0) {
    const char* e = getenv("CASMVS_TMA2_PER_SM");
    per_sm_env = e ? atoi(e) : 0;
  }
  const int smem_limit = (228 * 1024) / (C::kTotal + 1024);
  int per_sm = smem_limit < 2 ? smem_limit : 2;
  if (per_sm_env > 0 && per_sm_env < smem_limit) per_sm = per_sm_env;
  if (per_sm < 1) per_sm = 1;
  const int Dm = MODE == MODE_T ? p.Di : p.Do;
  const int Hm = MODE == MODE_T ? p.Hi : p.Ho, Wm = MODE == MODE_T ? p.Wi : p.Wo;
  p.tiles_w = (Wm + kTileW - 1) / kTileW;
  p.tiles_h = (Hm + kTileH - 1) / kTileH;
  const int nco = p.Cout / COUT;
  int cap = tma::pow2_floor(512 / per_sm) / C::GW;
  if (cap < 1) { per_sm = 1; cap = 512 / C::GW; }
  if (cap > 32) cap = 32;
  const long cols = (long)p.B * p.tiles_w * p.tiles_h;
  const int dchunk = tma::pick_dchunk(Dm, cap, cols, (long)num_sms() * per_sm / nco,
                                      MODE == MODE_S2 ? 2 : 1,
                                      MODE == MODE_S2 ? 1 : MODE == MODE_T ? 1 : 0);
  p.dchunk = dchunk;
  p.nchunks = (Dm + dchunk - 1) / dchunk;
  const long items = cols * p.nchunks;
  const ImageRef ir = image_cache_get(wpk, 2000 + MODE * 10000 + CIN * 100 + COUT,
                                      (size_t)C::kWBytes * nco, st);
  float* img = ir.img;
  if (!img) return -2;
  if (!ir.hit) {
    if constexpr (MODE == MODE_P5)
      build_image_p5_kernel<CIN, COUT><<<32, 256, 0, st>>>(wpk, img);
    else
      build_image_tma2_kernel<MODE, CIN, COUT><<<64, 256, 0, st>>>(wpk, img, p.Cout);
    if (int rc = after_launch("conv3d_tma2/build_image")) return rc;
    image_cache_built(img, st);
  }
  p.bimg = img;
  long resident = (long)num_sms() * per_sm / nco;
  if (resident < 1) resident = 1;
  const long gx = items < resident ? items : resident;
  tma::launch_pdl(ir.settled, kfn, dim3((unsigned)gx, (unsigned)nco), kThreads2, C::kTotal, st, *map, p);
  return after_launch("conv3d_tma2");
}

}  // namespace tma2

// Returns 0 when handled, 1 when the layer shape is left to the other kernels.
int conv3d_tma2(const float* x, const float* wpk, const float* scale, const float* shift,
                float slope, const float* skip, float* y, int B, int Cin, int Cout, int D, int h,
                int w, int kind, int stride, int precision_flags, cudaStream_t st) {
  const int precision = precision_flags & 0xff;
  static int enabled = -1;
  if (enabled < 0) {
    const char* e = getenv("CASMVS_TMA2");
    enabled = e ? atoi(e) : 3;                      // bit 0: stride-2, bit 1: transposed
  }
  if (!enabled || precision != CASMVS_TF32) return 1;
  if ((reinterpret_cast<uintptr_t>(x) & 15) != 0) return 1;
  tma2::Params p;
  p.scale = scale; p.shift = shift; p.skip = skip; p.y = y;
  p.slope = slope; p.B = B; p.Di = D; p.Hi = h; p.Wi = w; p.Cout = Cout;
  // every layer this kernel covers has Cout > 1: stored rounded unless the caller asks for fp32
  p.round_out = (precision_flags & CASMVS_KEEP_FP32_OUT) ? 0 : 1;
  if (kind == CASMVS_CONV && stride == 2 && (enabled & 1)) {
    if (skip) return 1;
    p.Do = (D - 1) / 2 + 1; p.Ho = (h - 1) / 2 + 1; p.Wo = (w - 1) / 2 + 1;
    if (Cin == 8 && Cout == 16) return tma2::launch2<tma2::MODE_S2, 8, 16>(x, wpk, p, st);
    if (Cin == 16 && Cout == 32) return tma2::launch2<tma2::MODE_S2, 16, 32>(x, wpk, p, st);
    if (Cin == 32 && Cout == 64) return tma2::launch2<tma2::MODE_S2, 32, 16>(x, wpk, p, st);
    return 1;
  }
  if (kind == CASMVS_CONV_TRANSPOSE && (enabled & 2)) {
    p.Do = 2 * D; p.Ho = 2 * h; p.Wo = 2 * w;
    if (Cin == 16 && Cout == 8) return tma2::launch2<tma2::MODE_T, 16, 8>(x, wpk, p, st);
    if (Cin == 32 && Cout == 16) return tma2::launch2<tma2::MODE_T, 32, 16>(x, wpk, p, st);
    if (Cin == 64 && Cout == 32) return tma2::launch2<tma2::MODE_T, 64, 8>(x, wpk, p, st);
    return 1;
  }
  return 1;
}

}  // namespace casmvs

using namespace casmvs;

extern "C" int casmvs_conv2d_5x5s2_fwd(const float* x, const float* w, const float* shift,
                                       float slope, float* y, int N, int Cin, int Cout, int H,
                                       int W, int round_tf32, void* stream) {
  CASMVS_REQUIRE(x && w && y, "conv2d_5x5s2: null pointer");
  CASMVS_REQUIRE(N >= 0 && H >= 2 && W >= 2, "conv2d_5x5s2: bad dims");
  CASMVS_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0, "conv2d_5x5s2: x must be 16 B aligned");
  if (N == 0) return 0;
  tma2::Params p;
  p.scale = nullptr; p.shift = shift; p.skip = nullptr; p.y = y; p.slope = slope;
  p.B = 1; p.Di = N; p.Hi = H; p.Wi = W; p.Do = N; p.Ho = (H - 1) / 2 + 1; p.Wo = (W - 1) / 2 + 1;
  p.Cout = Cout; p.round_out = round_tf32 ? 1 : 0;
  cudaStream_t st = as_stream(stream);
  if (Cin == 8 && Cout == 16) return tma2::launch2<tma2::MODE_P5, 8, 16>(x, w, p, st);
  if (Cin == 16 && Cout == 32) return tma2::launch2<tma2::MODE_P5, 16, 32>(x, w, p, st);
  set_error("conv2d_5x5s2: only the FeatureNet shapes 8->16 and 16->32 are built (got %d->%d)",
            Cin, Cout);
  return -1;
}
